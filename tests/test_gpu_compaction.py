"""Index.compact: the live rows move to the front of every plane, removed rows are purged, the scan covers only the
used slots (a device-side extent) and a slot -> id map keeps the ids.  An Index built from a device fp32 tensor keeps
that tensor as its master copy, so the tests hand compacted indexes a clone.

The yardstick is a fresh Index over the live rows: after compact() every route must answer exactly like it, with its
slots mapped to the ids, bit for bit -- and exactly like the same index before compact().  Captured graphs and the
serving pipeline follow a compaction without re-capture."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def _dev_db(n, D, seed):
    """Unit randn rows generated on the device (the R1M shape in seconds)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    db = torch.empty((n, D), dtype=torch.float32, device=DEV)
    for r0 in range(0, n, 65536):
        blk = torch.randn((min(65536, n - r0), D), device=DEV, generator=g)
        db[r0:r0 + blk.shape[0]] = blk / blk.norm(dim=1, keepdim=True)
    return db


def _planted(db, nq, seed, noise=0.3, rows=None):
    g = torch.Generator(device=DEV).manual_seed(seed)
    pool = torch.arange(db.shape[0], device=DEV) if rows is None else torch.as_tensor(rows, device=DEV)
    src = pool[torch.randperm(pool.numel(), generator=g, device=DEV)[:nq]]
    q = db[src] + noise * torch.randn((nq, db.shape[1]), generator=g, device=DEV) / db.shape[1] ** 0.5
    return (q / q.norm(dim=1, keepdim=True)).contiguous(), src.cpu().numpy()


def _remove_some(n, frac, seed):
    rs = np.random.RandomState(seed)
    return np.sort(rs.choice(n, int(round(frac * n)), replace=False)).astype(np.int64)


def _compact(m, db, removed, setup=None):
    """A fresh Index over the rows not in `removed` -> (index, live row numbers)."""
    keep = np.ones(db.shape[0], dtype=bool)
    keep[removed] = False
    rows = np.nonzero(keep)[0]
    ref = m.Index(db[torch.from_numpy(rows).to(db.device)].contiguous(), device=DEV)
    if setup:
        setup(ref)
    return ref, rows


def _mapped(s, i, rows):
    s, i = s.cpu().numpy(), i.cpu().numpy()
    return s, np.where(i >= 0, rows[np.maximum(i, 0)], -1)


def _np(res):
    return res[0].cpu().numpy(), res[1].cpu().numpy()


def _same(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# route -> (rows, D, queries, k, Index setup, search kwargs)
ROUTES = {
    "dense": (9000, 256, 70, 50, None, {}),
    "three": (200000, 256, 70, 100, lambda ix: setattr(ix, "fused", False), {}),
    "three_large_k": (200000, 256, 70, 1200, None, {}),
    "fused": (200000, 256, 70, 100, None, {}),
    "wide": (200000, 256, 300, 20, None, {"block_q": 1024}),
}


def _route_data(name):
    n, D, nq, k, setup, kw = ROUTES[name]
    db = _dev_db(n, D, 7)
    q, src = _planted(db, nq, 8)
    return db, q, src, k, setup, kw


def _bits(live):
    return np.unpackbits(live.cpu().numpy().view(np.uint8), bitorder="little").astype(bool)


# ---------------------------------------------------------------------------------------------------- 1. the kernel
@pytest.mark.parametrize("case", ["random", "head", "tail", "words", "none_live"])
@pytest.mark.parametrize("chunk", [100, 256, 1000])
def test_compaction_kernel_matches_numpy(m, case, chunk):
    """Every plane (bf16, fp32, int8, row_scale, slot -> id map) against numpy, the freed tail zero, the bitmap and the
    extent; capacity 3,001 (not a multiple of 32 or 256), chunks cut across bitmap words, staged and direct moves."""
    n_used, cap, D, base = 2900, 3001, 128, 70000
    db = _dev_db(n_used, D, 3)
    ix = m.Index(db, device=DEV, capacity=cap, idx_base=base)
    g = torch.Generator(device=DEV).manual_seed(4)
    ix.db8 = torch.zeros((cap, D), dtype=torch.int8, device=DEV)          # an int8 plane and scales to move along
    ix.db8[:n_used] = torch.randint(-127, 128, (n_used, D), generator=g, device=DEV, dtype=torch.int8)
    ix.row_scale = torch.zeros((cap,), dtype=torch.float32, device=DEV)
    ix.row_scale[:n_used] = torch.rand((n_used,), generator=g, device=DEV) + 0.5
    ix.compact_chunk = chunk
    rs = np.random.RandomState(5)
    removed = {"random": rs.choice(n_used, 1100, replace=False), "head": np.arange(0, 700), "tail": np.arange(2000, n_used),
               "words": np.concatenate([np.arange(31, 33), np.arange(255, 257), np.arange(992, 1024), [n_used - 1]]),
               "none_live": np.arange(n_used)}[case]
    ix.remove(removed + base)
    planes = [t.clone() for t in (ix.db16, ix.db32, ix.db8, ix.row_scale, ix.slot_id)]
    keep = np.setdiff1d(np.arange(n_used), removed)
    assert ix.compact() == len(removed)
    torch.cuda.synchronize()
    nl = len(keep)
    kd = torch.from_numpy(keep).to(DEV)
    for before, after in zip(planes, (ix.db16, ix.db32, ix.db8, ix.row_scale, ix.slot_id)):
        assert torch.equal(after[:nl], before[kd])
    for t in (ix.db16, ix.db32, ix.db8, ix.row_scale):
        assert not t[nl:].ne(0).any()
    assert (ix.slot_id[nl:n_used].cpu().numpy().view(np.uint32) == 0xffffffff).all()
    assert np.array_equal(ix.slot_id[:nl].cpu().numpy().view(np.uint32).astype(np.int64), keep + base)
    bits = _bits(ix.live)
    assert bits[:nl].all() and not bits[nl:].any()
    assert int(ix.n_scan.item()) == nl and ix.n_live == nl
    assert ix.compact() == 0                                            # nothing removed: a no-op


# ---------------------------------------------------------------------------------------------------- 2. scan extent
def _filter_candidates(m, ix, q16, tau_score, extent, wide):
    """One FILTER launch (no sample tiles, every row whose score reaches tau_score passes) over rows [0, extent) ->
    the candidate rows of every query."""
    lib, _lib = m.lib(), m._lib
    nq = q16.shape[0]
    rows = 256 if nq <= 256 else 1024
    tau = torch.full((rows,), int(lib.mdir_make_key(tau_score, 0xffffffff)), dtype=torch.int64, device=DEV)
    cand = torch.zeros((rows, m.search.CAND_ROW), dtype=torch.int64, device=DEV)
    cnt = torch.zeros((rows, m.search.N_SEGS), dtype=torch.int32, device=DEV)
    ext = torch.tensor([extent], dtype=torch.int64, device=DEV)
    fn = lib.mdir_sim_scan_wide_bf16_extent if wide else lib.mdir_sim_scan_bf16_extent
    _lib.check(fn(_lib.ptr(ix.db16), ix.n, _lib.ptr(q16), nq, ix.D, 2, 0, 0, None, 0, _lib.ptr(tau), 0, _lib.ptr(cand), _lib.ptr(cnt),
                  m.search.CAP_S, m.search.CAP_L, _lib.ptr(ix.live), _lib.ptr(ext), _lib.stream()), "scan")
    cand, cnt = cand.cpu().numpy(), cnt.cpu().numpy()
    out = []
    for j in range(nq):
        got = []
        for s in range(1, m.search.N_SEGS):
            c = int(cnt[j, s])
            assert c <= m.search.CAP_L
            off = m.search.CAP_S + (s - 1) * m.search.CAP_L
            got += [int(x) & 0xffffffff for x in cand[j, off:off + c]]
        out.append(sorted(got))
    return out


@pytest.mark.parametrize("wide", [False, True])
def test_filter_scan_stops_at_the_extent(m, wide):
    """Rows past the extent are live and are the best answers of every query: none of them may be a candidate."""
    n, D, extent = 60000, 256, 33333                      # the extent cuts a tile and a bitmap word
    nq = 300 if wide else 70
    db = _dev_db(n, D, 11)
    q = _dev_db(nq, D, 12)
    below = np.arange(nq) * 7 + 100                       # one planted row per query below the extent ...
    above = extent + np.arange(nq) * 11                   # ... and one past it, closer to the query
    db[torch.from_numpy(below).to(DEV)] = q
    db[torch.from_numpy(above).to(DEV)] = q
    ix = m.Index(db, device=DEV)
    q16 = m.search.pack_bf16(q)
    got = _filter_candidates(m, ix, q16, 0.5, extent, wide)
    assert got == [[int(b)] for b in below]
    full = _filter_candidates(m, ix, q16, 0.5, n, wide)   # without the bound both are found
    assert full == [sorted([int(b), int(a)]) for b, a in zip(below, above)]


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_fused_scan_stops_at_the_extent(m, precision):
    """The one-launch route with the extent set below the capacity equals a fresh index over the rows below it, although
    the planted answers of every query sit past it and are live."""
    n, D, nq, k, extent = 200000, 256, 70, 100, 120001
    db = _dev_db(n, D, 13)
    q, src = _planted(db, nq, 14, rows=np.arange(extent, n))
    ix = m.Index(db, device=DEV)
    assert ix._fused_ok(max(k, m.search.default_shortlist(k)), nq)
    ix.n_scan.fill_(extent)
    got = _np(ix.search(q, k, precision=precision))
    assert got[1].max() < extent
    ref = m.Index(db[:extent].contiguous(), device=DEV)
    assert _same(got, _np(ref.search(q, k, precision=precision)))


# ---------------------------------------------------------------------------------------------------- 3. equality
@pytest.mark.parametrize("frac", [0.01, 0.50, 0.90])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_compaction_equals_fresh_index(m, route, precision, frac):
    db, q, _, k, setup, kw = _route_data(route)
    removed = _remove_some(db.shape[0], frac, 11)
    index = m.Index(db.clone(), device=DEV)
    if setup:
        setup(index)
    index.remove(removed)
    before = _np(index.search(q, k, precision=precision, **kw))
    assert index.compact() == len(removed)
    after = _np(index.search(q, k, precision=precision, **kw))
    ref, rows = _compact(m, db, removed, setup)
    want = _mapped(*ref.search(q, k, precision=precision, **kw), rows)
    assert _same(before, want) and _same(after, want)
    assert int(index.n_scan.item()) == len(rows)


def test_fused_extent_below_the_grid_and_empty(m):
    """A fused launch over fewer used tiles than CTAs (CTAs without a sample tile), then over no tile at all."""
    db, q, _, k, _, _ = _route_data("fused")
    n = db.shape[0]
    keep = np.sort(np.random.RandomState(41).choice(n, 15000, replace=False))      # 59 tiles after compaction
    removed = np.setdiff1d(np.arange(n), keep)
    index = m.Index(db.clone(), device=DEV)
    index.remove(removed)
    index.compact()
    for precision in ("bf16", "fp32"):
        assert index._fused_ok(max(k, m.search.default_shortlist(k)), q.shape[0])
        ref, rows = _compact(m, db, removed)
        assert _same(_np(index.search(q, k, precision=precision)), _mapped(*ref.search(q, k, precision=precision), rows))
    index.remove(keep)
    assert index.compact() == len(keep) and int(index.n_scan.item()) == 0
    s, i = _np(index.search(q, k))
    assert (i == -1).all() and np.isneginf(s).all()


# ---------------------------------------------------------------------------------------------------- 4. lifecycle
def test_compact_add_remove_compact(m):
    """Ids stay monotone and are never reused; restoring a purged id raises, removing it is a no-op; after every step
    the index answers like a fresh one over its live rows."""
    n, D, nq, k, cap = 200000, 256, 70, 100, 210000
    base = 1000
    pool = _dev_db(n + 60000, D, 61)
    q, _ = _planted(pool, nq, 62)
    index = m.Index(pool[:n].clone(), device=DEV, capacity=cap, idx_base=base)
    rows = {base + r: r for r in range(n)}                # live id -> row of `pool`
    rs = np.random.RandomState(63)
    issued = n
    next_row = n

    def check():
        ids = np.array(sorted(rows), dtype=np.int64)
        ref = m.Index(pool[torch.from_numpy(np.array([rows[i] for i in ids])).to(DEV)].contiguous(), device=DEV)
        for precision in ("bf16", "fp32"):
            assert _same(_np(index.search(q, k, precision=precision)), _mapped(*ref.search(q, k, precision=precision), ids))
        assert np.array_equal(index.slot_id[:len(ids)].cpu().numpy().view(np.uint32).astype(np.int64), ids)

    for rnd in range(2):
        gone = rs.choice(sorted(rows), 40000 if rnd == 0 else 30000, replace=False)
        index.remove(gone)
        for g in gone:
            del rows[int(g)]
        assert index.compact() == len(gone)
        with pytest.raises(m.MdirError, match="purged"):
            index.restore(gone[:3])
        index.remove(gone[:3])                            # a no-op
        assert index.n_live == len(rows)
        check()
        add = 30000
        ids = index.add(pool[next_row:next_row + add]).numpy()
        assert np.array_equal(ids, np.arange(base + issued, base + issued + add))       # never reused
        for j, i in enumerate(ids):
            rows[int(i)] = next_row + j
        issued += add
        next_row += add
        check()
    assert int(index._ids.max()) >= base + cap                # ids run past idx_base + capacity
    with pytest.raises(m.MdirError, match="outside"):
        index.restore([base + issued])                        # past every id issued


def test_search_qe_after_compaction(m):
    from mdir_b200 import qe
    db, q, _, k, _, _ = _route_data("fused")
    removed = _remove_some(db.shape[0], 0.30, 61)
    index = m.Index(db.clone(), device=DEV)
    index.remove(removed)
    index.compact()
    ref, rows = _compact(m, db, removed)
    assert _same(_np(qe.search_qe(index, q, k)), _mapped(*qe.search_qe(ref, q, k), rows))


# ---------------------------------------------------------------------------------------------------- 5. graphs, pipeline
@pytest.mark.parametrize("split", [False, True])
def test_graph_captured_before_compaction(m, split):
    n, D, nq, k = 200000, 256, 70, 100
    db = _dev_db(n, D, 51)
    q, src = _planted(db, nq, 52)
    index = m.Index(db, device=DEV, capacity=n + 5000)
    gs = m.GraphedSearch(index, nq, k, overlap=split, split=split)
    assert gs.split == split

    def replay():
        s, i = gs(q)
        torch.cuda.synchronize()
        assert not gs.check_overflow()
        return _np((s, i))

    base = replay()
    removed = np.setdiff1d(_remove_some(n, 0.5, 53), src)
    index.remove(removed)
    index.compact()
    got = replay()
    ref, rows = _compact(m, db, removed)
    assert _same(got, _mapped(*ref.search(q, k), rows)) and _same(got, _np(index.search(q, k)))
    assert np.array_equal(got[1][:, 0], src)
    ids = index.add(q[:5])                                   # the queries themselves: their new top-1
    got = replay()
    assert np.array_equal(got[1][:5, 0], ids.numpy()) and _same(got, _np(index.search(q, k)))
    assert ids.numpy().min() == n                             # ids continue from the highest issued


def test_pipeline_compact(m):
    """compact() refuses while a ticket is pending; after collection it works, and later tickets -- one of them redone
    by the recovery path (hard queries whose certificate fails inside the graph) -- are exact."""
    n_db, D, n_q, k, dup = 100000, 128, 8, 100, 700
    rs = np.random.RandomState(9)
    db = synth.descriptors(n_db, D, 90)
    q_hard = synth.descriptors(n_q, D, 91)
    pos = rs.permutation(n_db)[:n_q * dup].reshape(n_q, dup)
    for j in range(n_q):
        nz = rs.randn(dup, D).astype(np.float32)
        nz -= (nz @ q_hard[j])[:, None] * q_hard[j][None, :]
        v = q_hard[j][None, :] + 0.1 * nz / np.sqrt(D)
        db[pos[j]] = v / np.linalg.norm(v, axis=1, keepdims=True)
    q_easy, _ = synth.planted_queries(synth.descriptors(n_db, D, 90), n_q, 92)
    index = m.Index(db, device=DEV)
    removed = np.setdiff1d(_remove_some(n_db, 0.4, 93), pos.ravel())
    pipe = m.SearchPipeline(index, n_q, k)
    hb = [torch.from_numpy(b).pin_memory() for b in (q_hard, q_easy)]
    t0 = pipe.submit(hb[1])
    pipe.remove(removed)
    with pytest.raises(m.MdirError, match="pending"):
        pipe.compact()
    pipe.result(t0)
    assert pipe.compact() == len(removed)
    ref, rows = _compact(m, torch.from_numpy(db).to(DEV), removed)
    want = [_mapped(*ref.search(torch.from_numpy(b).to(DEV), k), rows) for b in (q_hard, q_easy)]
    rec0 = pipe.n_recovered
    t1, t2 = pipe.submit(hb[0]), pipe.submit(hb[1])
    assert _same(pipe.result(t1), want[0]) and _same(pipe.result(t2), want[1])
    assert pipe.n_recovered == rec0 + 1                      # the hard batch went through the recovery path


# ---------------------------------------------------------------------------------------------------- R1M shape
@pytest.fixture(scope="module")
def r1m():
    n, D, nq = 1001001, 2048, 70
    db = _dev_db(n, D, 1234)
    q, src = _planted(db, nq, 99)
    yield db, q, src
    del db
    torch.cuda.empty_cache()


def test_r1m_int8_route_after_compaction(m, r1m):
    """70 q x 1,001,001 x 2048, k = 100, 50 % removed: the int8 first pass before and after compact() equals a fresh
    index over the live rows (which takes the bf16 route at 500 k rows)."""
    db, q, _ = r1m
    removed = _remove_some(db.shape[0], 0.50, 81)
    index = m.Index(db.clone(), device=DEV)
    index.remove(removed)
    before = _np(index.search(q, 100))
    assert index.route == "int8"
    index.compact()
    after = _np(index.search(q, 100))
    assert index.route == "int8" and index.cert["int8_redone"] == 0
    ref, rows = _compact(m, db, removed)
    want = _mapped(*ref.search(q, 100), rows)
    assert _same(before, want) and _same(after, want)
    del ref


def test_r1m_int8_scan_stops_at_the_extent(m, r1m):
    """The int8 fused scan with the extent at 600,000 rows: the planted answers past it are live but never returned."""
    db, _, _ = r1m
    extent = 600000
    q, _ = _planted(db, 70, 98, rows=np.arange(extent, db.shape[0]))
    index = m.Index(db, device=DEV)
    index.n_scan.fill_(extent)
    got = _np(index.search(q, 100))
    assert got[1].max() < extent
    ref = m.Index(db[:extent].contiguous(), device=DEV)
    assert _same(got, _np(ref.search(q, 100)))
    del ref


# ---------------------------------------------------------------------------------------------------- multi-GPU
def test_sharded_compaction_under_torchrun():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs: the sharded compaction path is not measured on one")
    world = 8 if n >= 8 else (4 if n >= 4 else 2)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", "29657", os.path.join(ROOT, "tools", "test_compaction_multi_gpu.py")]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900, cwd=ROOT)
    text = r.stdout.decode()
    assert r.returncode == 0 and "COMPACTION MULTI-GPU PASSED" in text and "[FAIL]" not in text, text[-6000:]
