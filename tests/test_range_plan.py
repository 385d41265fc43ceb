"""Host side of Index.range_search (no GPU): threshold validation, the CSR assembly of the gather's per-chunk survivor
counts, and the exact re-scan plan after a segment overflowed."""
import numpy as np
import pytest
import torch

from mdir_b200 import _lib
from mdir_b200.search import (RANGE_BUDGET, RANGE_CHUNK, range_chunks, range_csr, range_rescan_plan, range_thresholds)


def test_thresholds_broadcast_and_per_query():
    assert np.array_equal(range_thresholds(0.5, 3), np.full(3, 0.5, np.float32))
    assert range_thresholds(0.5, 0).shape == (0,)
    per = torch.tensor([0.1, -np.inf, np.inf], dtype=torch.float32)
    got = range_thresholds(per, 3)
    assert got.dtype == np.float32 and np.array_equal(got, per.numpy())
    assert np.array_equal(range_thresholds([1.0, 2.0], 2), np.array([1, 2], np.float32))


def test_thresholds_round_up_to_float32():
    # an fp32 score s passes s >= t (t float64) exactly when it passes s >= range_thresholds(t)
    rs = np.random.RandomState(0)
    t = np.concatenate([rs.randn(2000) * 0.3, [0.1, 1 / 3, -1 / 3, 1e-40, -1e-40, 0.0]])
    t32 = range_thresholds(t, t.size)
    assert (t32.astype(np.float64) >= t).all()
    below = np.nextafter(t32, np.float32(-np.inf))
    assert (below.astype(np.float64) < t).all()


def test_thresholds_refuse_nan_and_bad_shape():
    with pytest.raises(_lib.MdirError):
        range_thresholds(float("nan"), 2)
    with pytest.raises(_lib.MdirError):
        range_thresholds(torch.tensor([0.0, float("nan")]), 2)
    with pytest.raises(_lib.MdirError):
        range_thresholds([0.1, 0.2, 0.3], 2)
    with pytest.raises(_lib.MdirError):
        range_thresholds(np.zeros((2, 1)), 2)


def test_csr_from_run_lengths():
    rs = np.random.RandomState(1)
    run_len = rs.randint(0, RANGE_CHUNK + 1, size=(7, 28))
    run_len[2] = 0                                      # a query without results
    run_len[5, 3:] = 0
    counts, lims, run_off = range_csr(run_len)
    assert counts.dtype == np.int64 and lims.dtype == np.int64 and run_off.dtype == np.int32
    assert np.array_equal(counts, run_len.sum(1)) and counts[2] == 0
    assert lims[0] == 0 and np.array_equal(np.diff(lims), counts) and lims[-1] == run_len.sum()
    assert run_off.flags["C_CONTIGUOUS"]
    # chunk c of query q lands at [run_off[q, c], run_off[q, c] + run_len[q, c]) inside the query: a partition of [0, count)
    for q in range(run_len.shape[0]):
        cover = np.zeros(counts[q], dtype=int)
        for c in range(run_len.shape[1]):
            cover[run_off[q, c]:run_off[q, c] + run_len[q, c]] += 1
        assert (cover == 1).all()


def test_csr_empty():
    counts, lims, run_off = range_csr(np.zeros((0, 5), dtype=np.int32))
    assert counts.shape == (0,) and np.array_equal(lims, [0]) and run_off.shape == (0, 5)


def test_chunks_cover_a_candidate_row():
    for cap in (1, 32, 96, 192, 193, 7000):
        n = range_chunks(cap)
        assert n * RANGE_CHUNK >= 148 * cap > (n - 1) * RANGE_CHUNK


def test_rescan_plan_exact_capacity_and_budget():
    cap, group = range_rescan_plan(np.array([10, 250, 193]))
    assert cap == 256 and group == 3                    # the deepest segment, rounded up to 32; everything fits
    cap, group = range_rescan_plan(np.array([5]))
    assert cap == 32 and group == 1
    # min_score = -inf over 1,001,001 rows: every segment holds what its CTA scanned (~6,800 rows)
    max_seg = np.full(128, 6784)
    cap, group = range_rescan_plan(max_seg)
    per_query = 8 * (148 * cap + range_chunks(cap) * RANGE_CHUNK)
    assert cap >= 6784 and group * per_query <= RANGE_BUDGET < (group + 1) * per_query and 1 <= group < 128
    # a budget smaller than one query still plans one query per group (never zero)
    assert range_rescan_plan(max_seg, budget=1)[1] == 1
