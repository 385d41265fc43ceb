"""Mutable index: Index.remove / restore / add, a live-row bitmap read by every top-k route.

The yardstick is compaction: an index with some rows removed must answer exactly like a fresh Index over its live rows
(returned ids mapped back to slots), bit for bit, on every route -- dense, three-launch (sample -> select -> filter),
fused bf16, fused int8 and wide -- at both precisions.  Appending must reproduce a fresh Index over all rows, and CUDA
graphs / the serving pipeline must see each mutation in stream order without re-capture."""
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


def _planted(db, nq, seed, noise=0.3):
    g = torch.Generator(device=DEV).manual_seed(seed)
    src = torch.randperm(db.shape[0], generator=g, device=DEV)[:nq]
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


def _check_route(m, index, name, precision, k, nq):
    """The route the case is meant to exercise is the one search() takes."""
    kth = k if precision == "bf16" else max(k, m.search.default_shortlist(k))
    if name == "dense":
        assert index._route(kth, min(nq, 128))[0] == 0
    elif name in ("three", "three_large_k"):
        assert index._route(kth, min(nq, 128))[0] == 2
    elif name == "fused":
        assert index._fused_ok(kth, nq)


# ---------------------------------------------------------------------------------------------------- 1. update kernel
def test_live_update_kernel_matches_numpy(m):
    """mdir_live_update against numpy: set and clear, repeated ids, ids outside [idx_base, idx_base + capacity) ignored,
    word boundaries, a capacity that is not a multiple of 32."""
    lib, _lib = m.lib(), m._lib
    cap, base = 1000, 5000
    words = -(-cap // 256) * 8
    rs = np.random.RandomState(3)
    bits = np.zeros(words * 32, dtype=bool)
    live = torch.zeros((words,), dtype=torch.int32, device=DEV)

    def apply(ids, value):
        ids = np.asarray(ids, dtype=np.int64)
        d = torch.from_numpy(ids).to(DEV)
        _lib.check(lib.mdir_live_update(_lib.ptr(live), cap, base, _lib.ptr(d), len(ids), value, _lib.stream()), "mdir_live_update")
        r = ids - base
        r = r[(r >= 0) & (r < cap)]
        bits[r] = bool(value)
        got = np.unpackbits(live.cpu().numpy().view(np.uint8), bitorder="little").astype(bool)
        assert np.array_equal(got, bits)

    edges = [base + x for x in (0, 31, 32, 63, 64, 255, 256, 991, 992, 999)]
    apply(edges + edges + [base - 1, base + cap, base + cap + 31, 0, 2 ** 40], 1)
    apply(base + rs.randint(0, cap, 3000), 1)                         # many duplicates sharing words
    apply(base + rs.randint(0, cap, 700), 0)
    apply([base + 31, base + 32, base + 999, base + 999, base - 5, base + 1000], 0)
    apply(np.arange(base - 50, base + cap + 50), 1)
    assert not bits[cap:].any()                                       # the tail past the capacity never set
    apply(np.arange(base, base + cap, 2), 0)
    apply([], 1)


# ---------------------------------------------------------------------------------------------------- 2. removal == compaction
@pytest.mark.parametrize("frac", [0.01, 0.30])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_removal_equals_compaction(m, route, precision, frac):
    db, q, _, k, setup, kw = _route_data(route)
    removed = _remove_some(db.shape[0], frac, 11)
    index = m.Index(db, device=DEV)
    if setup:
        setup(index)
    _check_route(m, index, route, precision, k, q.shape[0])
    index.remove(torch.from_numpy(removed))
    assert index.n_live == db.shape[0] - len(removed)
    got = _np(index.search(q, k, precision=precision, **kw))
    assert index.status().eq(0).all()
    ref, rows = _compact(m, db, removed, setup)
    want = _mapped(*ref.search(q, k, precision=precision, **kw), rows)
    assert _same(got, want)
    assert not np.isin(got[1], removed).any()


# ---------------------------------------------------------------------------------------------------- 3. removing the answer
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_removing_the_answer_promotes_the_next_rows(m, precision):
    """Planted near-duplicates of each query are its top-k; removing them makes the next k rows the answer."""
    n, D, nq, k, dup = 200000, 256, 16, 10, 10
    db = _dev_db(n, D, 21)
    q = _dev_db(nq, D, 22)                                   # unrelated to the database rows
    g = torch.Generator(device=DEV).manual_seed(23)
    pos = torch.randperm(n, generator=g, device=DEV)[:nq * dup].view(nq, dup)
    for j in range(nq):
        v = q[j][None, :] + 0.02 * torch.randn((dup, D), generator=g, device=DEV) / D ** 0.5
        db[pos[j]] = v / v.norm(dim=1, keepdim=True)
    index = m.Index(db, device=DEV)
    s2, i2 = _np(index.search(q, 2 * k, precision=precision))
    assert set(i2[0, :dup].tolist()) == set(pos[0].cpu().numpy().tolist())
    index.remove(i2[:, :k].ravel())
    s1, i1 = _np(index.search(q, k, precision=precision))
    assert np.array_equal(i1, i2[:, k:]) and np.array_equal(s1, s2[:, k:])
    assert not np.isin(i1, i2[:, :k]).any()


# ---------------------------------------------------------------------------------------------------- 4. extremes
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("route", ["dense", "fused", "three"])
def test_extremes(m, route, precision):
    db, q, _, k, setup, kw = _route_data(route)
    n = db.shape[0]
    index = m.Index(db, device=DEV)
    if setup:
        setup(index)
    # 0 removed: the all-live bitmap gives exactly what the scan without a bitmap (NULL) gives
    base = _np(index.search(q, k, precision=precision, **kw))
    bitmap, index.live = index.live, None
    try:
        nul = _np(index.search(q, k, precision=precision, **kw))
    finally:
        index.live = bitmap
    assert _same(base, nul)
    # 90 % removed: the fused threshold may overflow the segments; the dense recovery answers exactly
    removed = _remove_some(n, 0.90, 31)
    index.remove(removed)
    got = _np(index.search(q, k, precision=precision, **kw))
    ref, rows = _compact(m, db, removed, setup)
    assert _same(got, _mapped(*ref.search(q, k, precision=precision, **kw), rows))
    # fewer live rows than k: every live row, then (-inf, -1) padding; status clear
    keep = np.sort(np.random.RandomState(32).choice(n, k // 2, replace=False))
    index.restore(keep)
    index.remove(np.setdiff1d(np.arange(n), keep))
    assert index.n_live == k // 2
    s, i = index.search(q, k, precision=precision, **kw)
    assert index.status().eq(0).all()
    s, i = s.cpu().numpy(), i.cpu().numpy()
    assert np.array_equal(np.sort(i[:, :k // 2], axis=1), np.tile(keep, (q.shape[0], 1)))
    assert (i[:, k // 2:] == -1).all() and np.isneginf(s[:, k // 2:]).all() and np.isfinite(s[:, :k // 2]).all()
    ref, rows = _compact(m, db, np.setdiff1d(np.arange(n), keep), setup)
    assert _same((s, i), _mapped(*ref.search(q, k, precision=precision, **kw), rows))
    # restore everything: bit-identical to the original
    index.restore(np.arange(n))
    assert index.n_live == n
    assert _same(_np(index.search(q, k, precision=precision, **kw)), base)


# ---------------------------------------------------------------------------------------------------- 5. append
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_append_equals_fresh_index(m, route, precision):
    """Index(db[:n0], capacity=n) + add() of the rest in chunks == Index(db): the bf16 and fp32 rows, the merged
    certificate stats and (int8 route) the new rows' int8 plane.  A search before the adds builds the stats first."""
    db, q, _, k, setup, kw = _route_data(route)
    n = db.shape[0]
    n0 = int(0.6 * n)
    index = m.Index(db[:n0].clone(), device=DEV, capacity=n)
    if setup:
        setup(index)
    assert index.n_live == n0 and index.n == n
    index.search(q, k, precision=precision, **kw)
    cuts = [n0, n0 + (n - n0) // 3, n0 + 2 * (n - n0) // 3, n]
    for a, b in zip(cuts[:-1], cuts[1:]):
        ids = index.add(db[a:b])
        assert np.array_equal(ids.numpy(), np.arange(a, b))
    assert index.n_live == n
    fresh = m.Index(db, device=DEV)
    if setup:
        setup(fresh)
    assert _same(_np(index.search(q, k, precision=precision, **kw)), _np(fresh.search(q, k, precision=precision, **kw)))
    if precision == "fp32":
        assert torch.equal(index.stats(), fresh.stats())
    with pytest.raises(m.MdirError):
        index.add(db[:1])


def test_capacity_and_id_errors(m):
    db = synth.descriptors(3000, 64, 41)
    index = m.Index(db, device=DEV, capacity=3100, idx_base=1000)
    assert index.n_live == 3000
    for bad in ([999], [4100], [1000, 5000]):
        with pytest.raises(m.MdirError):
            index.remove(bad)
    with pytest.raises(m.MdirError):
        index.restore([4000])                                # a free slot was never filled
    index.remove([1000, 1000, 1001])
    index.remove([1000])                                     # re-removing is a no-op
    assert index.n_live == 2998
    ids = index.add(db[:100])
    assert np.array_equal(ids.numpy(), np.arange(4000, 4100))
    index.restore([4000, 1000])
    assert index.n_live == 3099
    with pytest.raises(m.MdirError):
        index.add(db[:1])
    with pytest.raises(m.MdirError):
        m.Index(db, device=DEV, capacity=10)
    with pytest.raises(m.MdirError):
        m.Index(db, device=DEV, idx_base=2 ** 32 - 100)


# ---------------------------------------------------------------------------------------------------- 6. graphs, pipeline
@pytest.mark.parametrize("split", [False, True])
def test_graphed_search_sees_mutations_without_recapture(m, split):
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
    assert _same(base, _np(index.search(q, k)))
    assert np.array_equal(base[1][:, 0], src)
    removed = np.unique(base[1][:, :3].ravel())
    index.remove(removed)
    got = replay()
    ref, rows = _compact(m, db, removed)
    assert _same(got, _mapped(*ref.search(q, k), rows)) and _same(got, _np(index.search(q, k)))
    index.restore(removed)
    assert _same(replay(), base)
    ids = index.add(q[:5])                                   # the queries themselves: their new top-1
    got = replay()
    assert np.array_equal(got[1][:5, 0], ids.numpy()) and _same(got, _np(index.search(q, k)))


def test_pipeline_tickets_see_the_live_set_they_were_submitted_with(m):
    """Tickets in flight during a mutation answer with the old live set -- also when redone by the recovery path
    (hard queries whose certificate fails inside the graph) -- and tickets submitted after it with the new one."""
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
    index = m.Index(db, device=DEV, capacity=n_db + 64)
    before = [_np(index.search(b, k)) for b in (q_hard, q_easy)]
    removed = np.unique(np.concatenate([before[0][1][:, :20].ravel(), before[1][1][:, :20].ravel()]))
    other = m.Index(db, device=DEV, capacity=n_db + 64)
    other.remove(removed)
    after = [_np(other.search(b, k)) for b in (q_hard, q_easy)]
    new_ids = other.add(q_easy)
    added = [_np(other.search(b, k)) for b in (q_hard, q_easy)]
    assert np.array_equal(added[1][1][:, 0], new_ids.numpy())
    pipe = m.SearchPipeline(index, n_q, k)
    hb = [torch.from_numpy(b).pin_memory() for b in (q_hard, q_easy)]
    t0, t1 = pipe.submit(hb[0]), pipe.submit(hb[1])
    pipe.remove(removed)
    outs = [pipe.result(t0), pipe.result(t1)]
    assert all(_same(o, b) for o, b in zip(outs, before))
    t2, t3 = pipe.submit(hb[0]), pipe.submit(hb[1])
    pipe.add(q_easy)
    outs = [pipe.result(t2), pipe.result(t3)]
    assert all(_same(o, a) for o, a in zip(outs, after))
    t4, t5 = pipe.submit(hb[0]), pipe.submit(hb[1])
    outs = [pipe.result(t4), pipe.result(t5)]
    assert all(_same(o, a) for o, a in zip(outs, added))
    pipe.restore(removed)
    t6 = pipe.submit(hb[1])
    assert pipe.result(t6)[1][0, 0] == int(new_ids[0])
    assert pipe.n_recovered == 3                             # the hard batch of t0 (old live set), t2 and t4


# ---------------------------------------------------------------------------------------------------- 7. other operations
def test_search_qe_on_mutated_index_equals_compacted(m):
    from mdir_b200 import qe
    db, q, _, k, _, _ = _route_data("fused")
    removed = _remove_some(db.shape[0], 0.30, 61)
    index = m.Index(db, device=DEV)
    index.remove(removed)
    got = _np(qe.search_qe(index, q, k))
    ref, rows = _compact(m, db, removed)
    assert _same(got, _mapped(*qe.search_qe(ref, q, k), rows))


def test_dense_operations_refuse_dead_slots(m):
    from mdir_b200 import qe
    db = synth.descriptors(3000, 64, 71)
    q = synth.descriptors(4, 64, 72)
    for index in (m.Index(db, device=DEV, capacity=3001), m.Index(db, device=DEV)):
        if index.n == 3000:
            index.remove([5])
        for call in (lambda: index.scores(q), lambda: index.ranks(q), lambda: qe.dba(index)):
            with pytest.raises(m.MdirError, match="removed rows or free capacity"):
                call()
        index.search(q, 10)
    full = m.Index(db, device=DEV, capacity=3001)
    full.add(db[:1])
    assert full.scores(q).shape == (4, 3001)


# ---------------------------------------------------------------------------------------------------- R1M shape
@pytest.fixture(scope="module")
def r1m():
    n, D, nq = 1001001, 2048, 70
    db = _dev_db(n, D, 1234)
    q, src = _planted(db, nq, 99)
    yield db, q, src
    del db
    torch.cuda.empty_cache()


@pytest.mark.parametrize("frac", [0.01, 0.30])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_r1m_removal_equals_compaction(m, r1m, precision, frac):
    """The default route at the headline shape (fp32: the int8 first pass), 70 q x 1,001,001 x 2048, k = 100."""
    db, q, _ = r1m
    removed = _remove_some(db.shape[0], frac, 81)
    index = m.Index(db, device=DEV)
    index.remove(removed)
    got = _np(index.search(q, 100, precision=precision))
    if precision == "fp32":
        assert index.cert["int8_blocks"] == 1 and index.db8 is not None
    ref, rows = _compact(m, db, removed)
    assert _same(got, _mapped(*ref.search(q, 100, precision=precision), rows))
    del ref


def test_r1m_removal_against_fp64_ranking(m, r1m):
    """Independent check: the fp32 top-100 after removing 1 % equals the fp64 ranking of the live rows (indices may only
    differ between rows whose fp64 scores tie within fp32 rounding)."""
    db, q, _ = r1m
    removed = _remove_some(db.shape[0], 0.01, 82)
    index = m.Index(db, device=DEV)
    index.remove(removed)
    s, i = _np(index.search(q, 100))
    sc = (q.double() @ db.double().t())
    sc[:, torch.from_numpy(removed).to(DEV)] = -np.inf
    ref_s, ref_i = torch.topk(sc, 100, dim=1)
    ref_s, ref_i = ref_s.cpu().numpy(), ref_i.cpu().numpy()
    assert np.abs(s - ref_s).max() <= 3e-6
    diff = i != ref_i
    sc_np = sc.cpu().numpy() if diff.any() else None
    if diff.any():
        rq, cq = np.nonzero(diff)
        assert np.all(np.abs(sc_np[rq, i[rq, cq]] - sc_np[rq, ref_i[rq, cq]]) <= 4e-6)
    assert not np.isin(i, removed).any()


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_r1m_append_equals_fresh_index(m, r1m, precision):
    db, q, _ = r1m
    n = db.shape[0]
    n0 = 950000                                  # >= I8_MIN_ROWS filled: the int8 plane is built before the adds
    index = m.Index(db[:n0], device=DEV, capacity=n)
    index.search(q, 100, precision=precision)
    for a, b in ((n0, n0 + 20000), (n0 + 20000, n)):
        index.add(db[a:b])
    fresh = m.Index(db, device=DEV)
    assert _same(_np(index.search(q, 100, precision=precision)), _np(fresh.search(q, 100, precision=precision)))
    if precision == "fp32":
        assert index.route == fresh.route == "int8"
        assert torch.equal(index.stats(), fresh.stats())
        assert torch.equal(index.db8, fresh.db8) and torch.equal(index.row_scale, fresh.row_scale)


def test_r1m_split_graph_sees_mutations(m, r1m):
    """The split serving graphs (int8 scan | finalize + certified re-score) after remove / restore."""
    db, q, src = r1m
    index = m.Index(db, device=DEV)
    gs = m.GraphedSearch(index, q.shape[0], 100, overlap=True, split=True)
    assert gs.split
    base = _np(gs(q))
    torch.cuda.synchronize()
    assert np.array_equal(base[1][:, 0], src)
    removed = np.unique(base[1][:, :5].ravel())
    index.remove(removed)
    got = _np(gs(q))
    torch.cuda.synchronize()
    assert not gs.check_overflow()
    assert _same(got, _np(index.search(q, 100)))
    assert not np.isin(got[1], removed).any()
    index.restore(removed)
    assert _same(_np(gs(q)), base)


# ---------------------------------------------------------------------------------------------------- 8. multi-GPU
def test_sharded_remove_restore_under_torchrun():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 8 if n >= 8 else (4 if n >= 4 else 2)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", "29653", os.path.join(ROOT, "tools", "test_mutable_multi_gpu.py")]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900, cwd=ROOT)
    text = r.stdout.decode()
    assert r.returncode == 0 and "MUTABLE MULTI-GPU PASSED" in text and "[FAIL]" not in text, text[-6000:]
