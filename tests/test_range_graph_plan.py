"""Host side of captured range serving (no GPU): range_splice, the CSR splice of RangePipeline's recovery; the emit's
stage size; and the argument refusals of GraphedRangeSearch and RangePipeline that come before any device work."""
import numpy as np
import pytest

from mdir_b200 import _lib
from mdir_b200.search import (GraphedRangeSearch, Index, RangePipeline, ShardedIndex, range_splice, range_stage_cap)


def ragged_csr(rs, counts):
    """A CSR with these per-query counts: scores descending within a query, ids unique per query."""
    lims = np.zeros((len(counts) + 1,), np.int64)
    np.cumsum(counts, out=lims[1:])
    scores = np.concatenate([np.sort(rs.rand(c).astype(np.float32))[::-1] for c in counts] + [np.zeros(0, np.float32)])
    ids = np.concatenate([rs.choice(100000, c, replace=False).astype(np.int32) for c in counts] + [np.zeros(0, np.int32)])
    return lims, scores, ids


def direct(rows):
    """The CSR built directly from per-query (scores, ids) lists."""
    lims = np.zeros((len(rows) + 1,), np.int64)
    np.cumsum([s.size for s, _ in rows], out=lims[1:])
    return (lims, np.concatenate([s for s, _ in rows] + [np.zeros(0, np.float32)]),
            np.concatenate([i for _, i in rows] + [np.zeros(0, np.int32)]))


def rows_of(lims, scores, ids):
    return [(scores[a:b], ids[a:b]) for a, b in zip(lims[:-1], lims[1:])]


@pytest.mark.parametrize("case", ["random", "all", "none", "empty_queries", "empty_redo", "zero_queries"])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_splice_equals_direct_csr(case, seed):
    rs = np.random.RandomState(seed)
    nq = 0 if case == "zero_queries" else int(rs.randint(1, 40))
    counts = rs.randint(0, 50, size=nq)
    if case == "empty_queries":
        counts[::2] = 0
    flagged = {"random": np.flatnonzero(rs.rand(nq) < 0.3), "all": np.arange(nq), "none": np.zeros(0, np.int64),
               "empty_queries": np.flatnonzero(rs.rand(nq) < 0.5), "empty_redo": np.flatnonzero(rs.rand(nq) < 0.5),
               "zero_queries": np.zeros(0, np.int64)}[case]
    counts[flagged] = 0                              # the graph leaves a flagged query without rows
    base = ragged_csr(rs, counts)
    sub_counts = rs.randint(0, 80, size=flagged.size)
    if case == "empty_redo":
        sub_counts[::2] = 0                          # a flagged query whose redo is empty too
    sub = ragged_csr(rs, sub_counts)
    got = range_splice(*base, flagged, *sub)
    want_rows = rows_of(*base)
    for k, j in enumerate(flagged):
        want_rows[j] = rows_of(*sub)[k]
    want = direct(want_rows)
    for g, w in zip(got, want):
        assert g.dtype == w.dtype and np.array_equal(g, w)


def test_splice_replaces_rows_a_flagged_query_had():
    lims, scores, ids = np.array([0, 2, 3, 5]), np.array([5, 4, 3, 2, 1], np.float32), np.array([10, 11, 12, 13, 14], np.int32)
    got = range_splice(lims, scores, ids, [1], [0, 3], np.array([9, 8, 7], np.float32), np.array([20, 21, 22], np.int32))
    assert np.array_equal(got[0], [0, 2, 5, 7])
    assert np.array_equal(got[1], [5, 4, 9, 8, 7, 2, 1]) and np.array_equal(got[2], [10, 11, 20, 21, 22, 13, 14])


def test_splice_refuses_bad_arguments():
    lims, scores, ids = np.array([0, 1, 2]), np.zeros(2, np.float32), np.zeros(2, np.int32)
    e_s, e_i = np.zeros(0, np.float32), np.zeros(0, np.int32)
    with pytest.raises(_lib.MdirError):
        range_splice(lims, scores, ids, [1, 0], [0, 0, 0], e_s, e_i)     # not ascending
    with pytest.raises(_lib.MdirError):
        range_splice(lims, scores, ids, [2], [0, 0], e_s, e_i)           # no such query
    with pytest.raises(_lib.MdirError):
        range_splice(lims, scores, ids, [0], [0, 0, 0], e_s, e_i)        # sub_lims of the wrong length


def test_stage_cap():
    assert [range_stage_cap(m) for m in (1, 32, 33, 1000, 1024, 1025, 16384)] == [32, 32, 64, 1024, 1024, 2048, 16384]


def fake_index(keep_fp32):
    """An Index object that owns no device memory: enough for the refusals that precede any device work."""
    index = Index.__new__(Index)
    index.db32 = object() if keep_fp32 else None
    return index


@pytest.mark.parametrize("cls", [GraphedRangeSearch, RangePipeline])
def test_refusals_before_any_device_work(cls):
    with pytest.raises(_lib.MdirError):
        cls(ShardedIndex.__new__(ShardedIndex), 8)
    for n_q in (0, 129):
        with pytest.raises(_lib.MdirError):
            cls(fake_index(True), n_q)
    for max_results in (0, 16385):
        with pytest.raises(_lib.MdirError):
            cls(fake_index(True), 8, max_results=max_results)
    with pytest.raises(_lib.MdirError):
        cls(fake_index(False), 8)                                      # fp32 needs the master copy
    with pytest.raises(ValueError):
        cls(fake_index(True), 8, precision="fp16")


def test_pipeline_refuses_depth_zero():
    with pytest.raises(_lib.MdirError):
        RangePipeline(fake_index(True), 8, depth=0)
