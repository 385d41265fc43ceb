"""Captured range serving: GraphedRangeSearch and RangePipeline against eager Index.range_search.

An emitted query of the graph runs the same kernels in the same order as the eager route (pack, threshold keys, FILTER
scan, gather, emit), so its rows must equal range_search's bit for bit; only the CSR offsets come from the device
(mdir_range_offsets instead of the host's range_csr).  Flagged queries (a segment overflowed, or more matches than
max_results) have no rows in the graph's CSR, and RangePipeline redoes them eagerly: its result() must equal
range_search(check=True) for the whole batch.

The R1M-shape test is test_pipeline_r1m_shape (select it alone with -k r1m)."""
import numpy as np
import pytest
import torch

from test_gpu_range_search import build_case, kth_scores, ref64

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def host(lims, scores, ids):
    """A device CSR (full arenas allowed) -> packed numpy (lims, scores, ids)."""
    lims = lims.cpu().numpy()
    n = int(lims[-1])
    return lims, scores[:n].cpu().numpy(), ids[:n].cpu().numpy()


def assert_same(got, want, what=""):
    """Bit for bit: lims, score bits and ids."""
    assert np.array_equal(got[0], want[0]), what
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32)), what
    assert np.array_equal(got[2], want[2]), what


def graph_run(gr, q, thr):
    out = host(*gr(q, thr))
    return out, gr.status.cpu().numpy()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
def test_replay_equals_eager(m, dist, precision):
    """New queries and thresholds on every replay, no re-capture, eager search / range_search calls in between."""
    n_q, D = 24, 256
    db, q0 = build_case(dist, 60000, D, n_q, 21)
    index = m.Index(db, device=DEV)
    gr = m.GraphedRangeSearch(index, n_q, max_results=4096, precision=precision)
    for rep in range(3):
        q = q0
        if rep:
            g = torch.Generator(device=DEV).manual_seed(100 + rep)
            q = db[torch.randperm(db.shape[0], device=DEV, generator=g)[:n_q]] + 0.5 * torch.randn((n_q, D), device=DEV, generator=g) / D ** 0.5
            q = q / q.norm(dim=1, keepdim=True)
        ks = np.geomspace(3, 3000, n_q).astype(int)
        np.random.RandomState(rep).shuffle(ks)
        thr = kth_scores(ref64(db, q), ks).astype(np.float32)
        if dist == "near_dup" and rep == 0:
            thr[:] = 0.9
        got, status = graph_run(gr, q, thr)
        want = host(*index.range_search(q, torch.from_numpy(thr), precision=precision))
        assert not status.any() and not gr.check_overflow()
        assert_same(got, want, (dist, precision, rep))
        # eager calls between replays change nothing in the graph's result, and the graph nothing in theirs
        s1, i1 = index.search(q, 50, precision=precision)
        index.range_search(q[:5], float("-inf"), precision=precision)
        again = host(gr.lims, gr.scores, gr.ids)
        assert_same(again, got)
        assert_same(host(*index.range_search(q, torch.from_numpy(thr), precision=precision)), want)
        gr()
        s2, i2 = index.search(q, 50, precision=precision)
        assert torch.equal(s1, s2) and torch.equal(i1, i2)
        assert_same(host(gr.lims, gr.scores, gr.ids), got)


def test_replay_equals_eager_d2048(m):
    n_q, D = 70, 2048
    db, q = build_case("randn", 60000, D, n_q, 22)
    index = m.Index(db, device=DEV)
    gr = m.GraphedRangeSearch(index, n_q, max_results=1024)
    thr = kth_scores(ref64(db, q), np.geomspace(5, 1000, n_q).astype(int)).astype(np.float32)
    got, status = graph_run(gr, q, thr)
    assert not status.any()
    assert_same(got, host(*index.range_search(q, torch.from_numpy(thr))))


def test_offsets_kernel_equals_range_csr(m):
    """mdir_range_offsets on the gather's real outputs (an eager check=False pass, which leaves them in the route's
    buffers) against range_csr, masked to the emitted queries, for several max_results."""
    from mdir_b200 import _lib
    from mdir_b200.search import MAX_Q, RANGE_CAP_L, range_chunks, range_csr
    n_q, D = 40, 128
    db, q = build_case("clusters", 100000, D, n_q, 23)
    index = m.Index(db, device=DEV)
    thr = kth_scores(ref64(db, q), np.geomspace(1, 20000, n_q).astype(int)).astype(np.float32)
    thr[3] = -np.inf                                    # segments overflow
    thr[7] = 2.0                                        # nothing
    index.range_search(q, torch.from_numpy(thr), check=False)
    n_chunks = range_chunks(RANGE_CAP_L)
    runs = index._buf("range_runs", (MAX_Q * (n_chunks + 1),), torch.int32)
    run_len, max_seg = runs[:n_q * n_chunks], runs[n_q * n_chunks:n_q * (n_chunks + 1)]
    rl_h, ms_h = run_len.cpu().numpy().reshape(n_q, n_chunks), max_seg.cpu().numpy()
    counts, _, run_off_h = range_csr(rl_h)
    assert (ms_h > RANGE_CAP_L).any() and (counts > 1024).any()
    for max_results in (1, 100, 1024, 16384):
        lims = torch.full((n_q + 1,), -7, dtype=torch.int64, device=DEV)
        run_off = torch.full((n_q, n_chunks), -7, dtype=torch.int32, device=DEV)
        status = torch.full((n_q,), -7, dtype=torch.int32, device=DEV)
        _lib.check(_lib.lib().mdir_range_offsets(_lib.ptr(run_len), _lib.ptr(max_seg), n_q, n_chunks, RANGE_CAP_L, max_results,
                                                 _lib.ptr(lims), _lib.ptr(run_off), _lib.ptr(status), _lib.stream()), "mdir_range_offsets")
        want_status = np.where(ms_h > RANGE_CAP_L, 1, 0) | np.where(counts > max_results, 8, 0)
        emitted = np.where(want_status == 0, counts, 0)
        want_lims = np.concatenate([[0], np.cumsum(emitted)])
        assert np.array_equal(status.cpu().numpy(), want_status), max_results
        assert np.array_equal(lims.cpu().numpy(), want_lims), max_results
        assert np.array_equal(run_off.cpu().numpy(), run_off_h), max_results


def mixed_case(m, n_q=8):
    D, n = 128, 100000
    db, q = build_case("randn", n, D, n_q, 24)
    index = m.Index(db, device=DEV)
    ref = ref64(db, q)
    thr = kth_scores(ref, np.full(n_q, 60)).astype(np.float32)
    thr[2] = np.float32(np.sort(ref[2])[::-1][1500])    # more matches than max_results, no segment overflow
    thr[4] = -np.inf                                    # every row: segments overflow
    thr[6] = 2.0                                        # above every score
    return index, db, q, thr


def test_mixed_batch_flags_and_pipeline_recovers(m):
    index, _, q, thr = mixed_case(m)
    gr = m.GraphedRangeSearch(index, q.shape[0], max_results=256)
    (lims, sc, ids), status = graph_run(gr, q, thr)
    assert status[2] == 8                               # STATUS_RANGE_FULL only
    assert status[4] & 1                                # STATUS_OVERFLOW
    assert (status[[0, 1, 3, 5, 6, 7]] == 0).all()
    counts = np.diff(lims)
    assert counts[2] == 0 and counts[4] == 0 and counts[6] == 0 and (counts[[0, 1, 3, 5, 7]] > 0).all()
    want = host(*index.range_search(q, torch.from_numpy(thr)))
    want_rows = [(want[1][a:b], want[2][a:b]) for a, b in zip(want[0][:-1], want[0][1:])]
    for j in (0, 1, 3, 5, 7):
        a, b = lims[j], lims[j + 1]
        assert np.array_equal(sc[a:b].view(np.uint32), want_rows[j][0].view(np.uint32)) and np.array_equal(ids[a:b], want_rows[j][1])
    pipe = m.RangePipeline(index, q.shape[0], max_results=256)
    qh = q.cpu()
    got = pipe.result(pipe.submit(qh, thr))
    assert_same(got, want)
    assert pipe.n_recovered == 1 and pipe.recovered["range_full"] >= 1 and pipe.recovered["overflow"] >= 1
    assert np.diff(got[0])[4] == 100000


def test_writes_stay_inside_the_arena(m):
    """No sanitizer: the arenas are filled with a sentinel before a replay.  Every position of [0, lims[n_q]) is
    written exactly once (no sentinel left, ids unique and sorted within each query) and nothing past lims[n_q] is
    touched, with flagged queries in the batch."""
    index, _, q, thr = mixed_case(m)
    gr = m.GraphedRangeSearch(index, q.shape[0], max_results=256)
    sentinel = -0x5A5A5A5A
    gr.scores.view(torch.int32).fill_(sentinel)
    gr.ids.fill_(sentinel)
    gr(q, thr)
    lims = gr.lims.cpu().numpy()
    sc_bits, ids = gr.scores.view(torch.int32).cpu().numpy(), gr.ids.cpu().numpy()
    sc = gr.scores.cpu().numpy()
    n = int(lims[-1])
    assert 0 < n < sc.size
    assert (sc_bits[n:] == sentinel).all() and (ids[n:] == sentinel).all()
    assert (sc_bits[:n] != sentinel).all() and (ids[:n] >= 0).all()
    for a, b in zip(lims[:-1], lims[1:]):
        assert np.unique(ids[a:b]).size == b - a
        assert (np.diff(sc[a:b]) <= 0).all()


def test_mutations_without_recapture(m):
    D, n0, cap, n_q = 128, 50000, 60000, 16
    db, q = build_case("randn", n0, D, n_q, 25)
    index = m.Index(db, device=DEV, capacity=cap)
    gr = m.GraphedRangeSearch(index, n_q, max_results=2048)
    gr_bf = m.GraphedRangeSearch(index, n_q, max_results=2048, precision="bf16")
    thr = 0.2

    def check(what):
        """Both graphs against eager range_search -> the fp32 result."""
        out = {}
        for g, p in ((gr, "fp32"), (gr_bf, "bf16")):
            out[p], status = graph_run(g, q, thr)
            assert not status.any(), what
            assert_same(out[p], host(*index.range_search(q, thr, precision=p)), (what, p))
        return out["fp32"]

    base = check("base")
    found = np.unique(base[2])
    rs = np.random.RandomState(0)
    gone = np.concatenate([found[::3], rs.choice(n0, 5000, replace=False)])
    index.remove(gone)
    after = check("remove")
    assert not set(after[2].tolist()) & set(gone.tolist())
    index.restore(gone)
    assert_same(check("restore"), base)
    # add into free capacity after capture: rows of norm 1.5 raise the certificate's bound (the stats grow in place)
    eps0 = index.stats().clone()
    new = 1.5 * (q + 0.05 * torch.randn(q.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(7)) / D ** 0.5)
    new_ids = index.add(new).numpy()
    assert (index.stats() > eps0).any()
    added = check("add")
    lims = added[0]
    for j in range(n_q):
        assert added[2][lims[j]] == new_ids[j]          # the scaled near-copy is the best match
    index.remove(np.concatenate([found[1::4], rs.choice(n0, 20000, replace=False), new_ids[::5]]))
    before = check("remove 2")
    assert index.compact() > 0
    assert_same(check("compact"), before)
    # every row removed and compacted: an empty CSR
    index.remove(index._ids.copy())
    assert index.compact() > 0
    got = check("empty")
    assert (got[0] == 0).all() and got[1].size == 0


def test_pipeline_mutations_and_inflight_bitmap(m):
    D, n0, cap, n_q = 128, 50000, 60000, 8
    db, q = build_case("randn", n0, D, n_q, 26)
    index = m.Index(db, device=DEV, capacity=cap)
    pipe = m.RangePipeline(index, n_q, max_results=512, depth=3)
    thr = np.full(n_q, 0.2, np.float32)
    thr[5] = -np.inf                                     # flagged every time: the ticket is recovered eagerly
    qh = q.cpu().pin_memory()
    before = host(*index.range_search(q, torch.from_numpy(thr)))
    found = np.unique(before[2][before[0][0]:before[0][5]])
    gone = np.concatenate([found[::2], np.arange(0, n0, 3)])
    t0 = pipe.submit(qh, thr)
    pipe.remove(gone)                                    # t0 keeps the bitmap it was submitted with, also in recovery
    t1 = pipe.submit(qh, thr)
    with pytest.raises(m.MdirError):
        pipe.compact()                                   # tickets pending
    r0 = pipe.result(t0)
    assert_same(r0, before)
    removed = host(*index.range_search(q, torch.from_numpy(thr)))
    assert_same(pipe.result(t1), removed)
    assert pipe.n_recovered == 2
    pipe.restore(gone[::2])
    new_ids = pipe.add(1.5 * q).numpy()
    assert pipe.compact() > 0
    want = host(*index.range_search(q, torch.from_numpy(thr)))
    outs = list(pipe.map([(qh, thr)] * 5))
    for o in outs:
        assert_same(o, want)
    lims = want[0]
    for j in (0, 1, 2, 3, 4, 6, 7):
        assert want[2][lims[j]] == new_ids[j]
    # every row removed and compacted: empty results (the -inf query too: no segment holds anything)
    pipe.remove(index._ids.copy())
    pipe.compact()
    got = pipe.result(pipe.submit(qh, thr))
    assert (got[0] == 0).all() and got[1].size == 0


def test_pipeline_r1m_shape(m):
    """1,001,001 x 2048, 70 queries: a few batches at ~100 and ~1,000 matches per query through the pipeline, equal to
    eager range_search."""
    n_db, D, nq = 1001001, 2048, 70
    g = torch.Generator(device=DEV).manual_seed(27)
    db = torch.empty((n_db, D), dtype=torch.float32, device=DEV)
    for r0 in range(0, n_db, 65536):
        r1 = min(n_db, r0 + 65536)
        blk = torch.randn((r1 - r0, D), device=DEV, generator=g)
        db[r0:r1] = blk / blk.norm(dim=1, keepdim=True)
    index = m.Index.from_packed(m.search.pack_bf16(db), db32=db)
    batches = []
    for b in range(4):
        src = torch.randperm(n_db, device=DEV, generator=g)[:nq]
        q = db[src] + 0.5 * torch.randn((nq, D), device=DEV, generator=g) / D ** 0.5
        q = q / q.norm(dim=1, keepdim=True)
        k = 100 if b % 2 == 0 else 1000
        s, _ = index.search(q, k)
        batches.append((q.cpu().pin_memory(), s[:, k - 1].cpu().numpy()))
    pipe = m.RangePipeline(index, nq, max_results=2048)
    for (q, thr), got in zip(batches, pipe.map(batches)):
        want = host(*index.range_search(q, thr))
        assert_same(got, want)
    print("R1M range pipeline: %d tickets, %d recovered %s" % (len(batches), pipe.n_recovered, pipe.recovered))
