"""GraphedDiffusion and DiffusionPipeline on the GPU: replays equal Diffusion.search / DiffusionTable.search bit for bit
(flagged queries: no rows and their status words); the graphs survive add / remove / restore / compact made through
the Diffusion without re-capture; stale sources are refused; the pipeline redoes flagged queries, settles pending
tickets before a mutation and refuses every mutation of a table."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_diffusion import build_case  # noqa: E402
from oracle import synth  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N_DB, D, K = 20000, 128, 50
WIDTH, TRUNC = 100, 500
PARAMS = dict(alpha=0.99, iters=20, rtol=1e-6)


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def _unit(x):
    return x / x.norm(dim=1, keepdim=True)


def noisy_rows(db, n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    src = torch.randint(0, db.shape[0], (n,), device=DEV, generator=g)
    return _unit(db[src] + 0.5 * torch.randn((n, db.shape[1]), device=DEV, generator=g) / db.shape[1] ** 0.5)


_CASES = {}


def case(m, dist):
    """(index, Diffusion(k=50), table(width 100, trunc 500), Q (256, D)), built once per module.  Q's rows 0..7 and
    128..135 are build_case's queries (near_dup: the ones with 200 near-duplicates each), the rest noisy database rows."""
    if dist not in _CASES:
        db, q = build_case(dist)
        index = m.Index(db, device=DEV)
        g = m.Diffusion(index, k=K, gamma=3.0)
        Q = noisy_rows(db, 256, 3)
        Q[:8] = q
        Q[128:136] = q.flip(0)
        _CASES[dist] = (index, g, g.offline(width=WIDTH, trunc=TRUNC, **PARAMS), Q)
    return _CASES[dist]


def raw_status(index, q, depth):
    """The status words of the shortlist search the graph runs (check=False: no widening, no recovery)."""
    index.search(q, depth, precision="fp32", check=False)
    return index.status()[:q.shape[0]].clone()


def assert_replay(f, ids, st, ef, eids, est):
    """Replay (f, ids, st) against the eager result (ef, eids) and the raw status words est: equal status words, rows
    with word 0 equal bit for bit, flagged rows all -inf / -1.  Returns the number of flagged rows."""
    f, ids, st, ef, eids, est = (t.cpu() for t in (f, ids, st, ef, eids, est))
    assert torch.equal(st, est)
    ok = st == 0
    assert torch.equal(f[ok].view(torch.int32), ef[ok].view(torch.int32)) and torch.equal(ids[ok], eids[ok])
    assert (ids[~ok] == -1).all() and torch.isneginf(f[~ok]).all()
    return int((~ok).sum())


def replay_twice(m, src, index, Q, n_q, k, p, depth):
    """Capture once; replay two query batches, with eager calls on the same stream between the replays."""
    gd = m.GraphedDiffusion(src, n_q, k, **p)
    flagged = 0
    for qb in (Q[:n_q], Q[128:128 + n_q]):
        f, ids = gd(qb)
        f, ids, st = f.clone(), ids.clone(), gd.status.clone()
        ef, eids = src.search(qb, k=k, **p)                              # eager, on the replay's stream
        flagged += assert_replay(f, ids, st, ef, eids, raw_status(index, qb, depth))
        assert torch.equal(gd.f.view(torch.int32), f.view(torch.int32)) and torch.equal(gd.ids, ids)   # eager calls leave it
    return flagged


# ------------------------------------------------------------------------------------------------- 1. replay == eager
@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
@pytest.mark.parametrize("k,trunc,k_q", [(100, 1000, 10), (2048, 2048, 10), (7, 64, 64)])
@pytest.mark.parametrize("n_q", [1, 70, 128])
def test_online_replay_equals_eager(m, dist, k, trunc, k_q, n_q):
    index, g, _, Q = case(m, dist)
    replay_twice(m, g, index, Q, n_q, k, dict(trunc=trunc, k_q=k_q, **PARAMS), trunc)


@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
@pytest.mark.parametrize("k,k_q", [(100, 10), (8192, 81)])
@pytest.mark.parametrize("n_q", [1, 70, 128])
def test_table_replay_equals_eager(m, dist, k, k_q, n_q):
    index, _, tab, Q = case(m, dist)
    replay_twice(m, tab, index, Q, n_q, k, dict(k_q=k_q), k_q)


# ------------------------------------------------------------------------------- 2. graphs survive updates, no re-capture
def test_graph_survives_updates_through_the_diffusion(m):
    db, _ = build_case("clusters", seed=5)
    n0 = 18000
    index = m.Index(db[:n0].clone(), device=DEV, capacity=N_DB)
    g = m.Diffusion(index, k=K, gamma=3.0)
    p = dict(trunc=1000, k_q=10, **PARAMS)
    q = noisy_rows(db[:n0], 70, 8)
    gd = m.GraphedDiffusion(g, 70, 100, **p)
    pipe = m.DiffusionPipeline(g, 70, 100, **p)

    def check(dif):
        f, ids = gd(q)
        ef, eids = dif.search(q, k=100, **p)
        n_flag = assert_replay(f, ids, gd.status, ef, eids, raw_status(index, q, 1000))
        pf, pids = pipe.result(pipe.submit(q.cpu()))
        assert np.array_equal(pf.view(np.int32), ef.cpu().numpy().view(np.int32)) and np.array_equal(pids, eids.cpu().numpy())
        return ids.clone(), n_flag

    ids0, _ = check(g)
    # rows just next to the queries: they become the queries' top results, and n_used grows past the captured count
    near = _unit(q + 0.05 * torch.randn(q.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(4)) / D ** 0.5)
    new = g.add(torch.cat([near, db[n0:n0 + 1000]]))
    assert index._n_used == n0 + 1070
    ids1, _ = check(g)
    assert np.array_equal(index.search(q, 1)[1][:, 0].cpu().numpy(), new.numpy()[:70])    # each query's shortlist leads with one
    gone = np.unique(np.concatenate([ids1.cpu().numpy()[:, :5].ravel(), np.arange(0, n0, 7)]))
    g.remove(gone)
    check(g)
    g.restore(gone[::2])
    check(g)
    assert g.compact() > 0
    ids_c, _ = check(g)
    fresh = m.Diffusion(index, k=K, gamma=3.0)                             # a new graph over the final index
    ef, eids = fresh.search(q, k=100, **p)
    f, ids = gd(q)
    ok = (gd.status == 0).cpu()
    assert torch.equal(f.cpu()[ok].view(torch.int32), ef.cpu()[ok].view(torch.int32)) and torch.equal(ids.cpu()[ok], eids.cpu()[ok])
    assert not np.isin(ids_c.cpu().numpy(), np.setdiff1d(gone, gone[::2])).any()


# ----------------------------------------------------------------------------------------------- 3. stale sources refused
def test_stale_sources_are_refused(m):
    db, q = build_case("randn", seed=9)
    index = m.Index(db[:5000], device=DEV, capacity=6000)
    g = m.Diffusion(index, k=20)
    tab = g.offline(width=50, trunc=200, **PARAMS)
    go = m.GraphedDiffusion(g, 8, 50, trunc=200, k_q=10, **PARAMS)
    gt = m.GraphedDiffusion(tab, 8, 50, k_q=10)
    po = m.DiffusionPipeline(g, 8, 50, trunc=200, k_q=10, **PARAMS)
    pt = m.DiffusionPipeline(tab, 8, 50, k_q=10)
    go(q), gt(q)
    po.result(po.submit(q)), pt.result(pt.submit(q))
    g.add(db[5000:5010])                                                   # through the Diffusion: the graph follows
    go(q)
    po.result(po.submit(q))
    with pytest.raises(m.MdirError, match="offline"):                      # the table does not
        gt(q)
    with pytest.raises(m.MdirError, match="offline"):
        pt.submit(q)
    index.remove([5])                                                      # on the index directly: everything is stale
    with pytest.raises(m.MdirError, match="mutated"):
        go(q)
    with pytest.raises(m.MdirError, match="mutated"):
        po.submit(q)
    index.compact()
    tab2 = m.Diffusion(index, k=20).offline(width=50, trunc=200, **PARAMS)
    pt2 = m.DiffusionPipeline(tab2, 8, 50, k_q=10)
    t = pt2.submit(q)
    for fn in (lambda: pt2.add(db[5010:5011]), lambda: pt2.remove([7]), lambda: pt2.restore([5]), pt2.compact):
        with pytest.raises(m.MdirError):
            fn()
    pt2.result(t)
    for fn in (lambda: pt2.add(db[5010:5011]), lambda: pt2.remove([7]), lambda: pt2.restore([5]), pt2.compact):
        with pytest.raises(m.MdirError, match="offline"):
            fn()
    assert index._n_used == 5009 and index.n_live == 5009                  # nothing was mutated


# ------------------------------------------------------------------------------------------------- 4. flagged queries
_HARD = {}


def hard_case(m):
    """100,000 x 128 rows with 700 near-duplicates around each of 8 hard queries: more than a 100-row shortlist (or a
    10-row top-k_q) can certify inside the graph.  (index with 64 free slots, Diffusion, table, hard + easy batch,
    easy-only batch)."""
    if not _HARD:
        n_db, n_q, dup = 100000, 8, 700
        rs = np.random.RandomState(9)
        db = synth.descriptors(n_db, D, 90)
        q_hard = synth.descriptors(n_q, D, 91)
        pos = rs.permutation(n_db)[:n_q * dup].reshape(n_q, dup)
        for j in range(n_q):
            nz = rs.randn(dup, D).astype(np.float32)
            nz -= (nz @ q_hard[j])[:, None] * q_hard[j][None, :]
            v = q_hard[j][None, :] + 0.1 * nz / np.sqrt(D)
            db[pos[j]] = v / np.linalg.norm(v, axis=1, keepdims=True)
        q_easy, _ = synth.planted_queries(synth.descriptors(n_db, D, 90), 3 * n_q, 92)
        index = m.Index(db, device=DEV, capacity=n_db + 64)
        g = m.Diffusion(index, k=K, gamma=3.0)
        tab = g.offline(width=WIDTH, trunc=TRUNC, **PARAMS)
        _HARD.update(index=index, g=g, tab=tab, batch=torch.from_numpy(np.concatenate([q_hard, q_easy[:n_q]])).pin_memory(),
                     easy=torch.from_numpy(q_easy[n_q:]).pin_memory(), extra=q_easy[:n_q])     # batches of 16 queries
    return _HARD


@pytest.mark.parametrize("online", [True, False])
def test_flagged_queries_replay_and_pipeline(m, online):
    h = hard_case(m)
    index, batch = h["index"], h["batch"]
    src, p, depth = (h["g"], dict(trunc=100, k_q=10, **PARAMS), 100) if online else (h["tab"], dict(k_q=10), 10)
    ef, eids = src.search(batch, k=100, **p)
    gd = m.GraphedDiffusion(src, 16, 100, **p)
    f, ids = gd(batch)
    est = raw_status(index, batch.to(DEV), depth)
    n_flag = assert_replay(f, ids, gd.status, ef, eids, est)
    assert n_flag >= 4 and (est[8:] == 0).all()                             # the hard queries, and only those
    pipe = m.DiffusionPipeline(src, 16, 100, **p)
    outs = list(pipe.map([batch, h["easy"], batch]))
    for (pf, pids), qb in zip(outs, [batch, h["easy"], batch]):
        wf, wids = src.search(qb, k=100, **p)
        assert np.array_equal(pf.view(np.int32), wf.cpu().numpy().view(np.int32)) and np.array_equal(pids, wids.cpu().numpy())
    st = est.cpu().numpy()
    assert pipe.n_recovered == 2
    assert pipe.recovered["overflow"] == 2 * int(((st & 1) != 0).sum()) and pipe.recovered["uncertified"] == 2 * int(((st & 2) != 0).sum())


# ------------------------------------------------------------------------------------------------- 5. pipeline ordering
def _np(t):
    return t[0].cpu().numpy(), t[1].cpu().numpy()


def _same(a, b):
    return np.array_equal(a[0].view(np.int32), b[0].view(np.int32)) and np.array_equal(a[1], b[1])


def test_pipeline_tickets_see_the_graph_they_were_submitted_under(m):
    h = hard_case(m)
    g, batch, easy = h["g"], h["batch"], h["easy"]
    p = dict(trunc=100, k_q=10, **PARAMS)
    pipe = m.DiffusionPipeline(g, 16, 100, depth=3, **p)
    before = [_np(g.search(b, k=100, **p)) for b in (batch, easy)]
    removed = np.unique(np.concatenate([before[0][1][8:, :10].ravel(), before[1][1][:, :10].ravel()]))
    removed = removed[removed >= 0]
    t0, t1 = pipe.submit(batch), pipe.submit(easy)                          # t0: a hard batch, settled by remove()
    pipe.remove(removed)
    assert pipe.n_recovered == 1
    after = [_np(g.search(b, k=100, **p)) for b in (batch, easy)]
    assert not _same(after[1], before[1])
    t2 = pipe.submit(batch)
    assert _same(pipe.result(t0), before[0]) and _same(pipe.result(t1), before[1])
    assert _same(pipe.result(t2), after[0])
    t3, t4 = pipe.submit(batch), pipe.submit(easy)
    new_ids = pipe.add(h["extra"])                                         # rows equal to the easy half of the batch
    added = [_np(g.search(b, k=100, **p)) for b in (batch, easy)]
    assert not _same(added[0], after[0])
    t5 = pipe.submit(batch)
    assert _same(pipe.result(t3), after[0]) and _same(pipe.result(t4), after[1]) and _same(pipe.result(t5), added[0])
    t6 = pipe.submit(easy)
    pipe.restore(removed)
    restored = _np(g.search(easy, k=100, **p))
    t7 = pipe.submit(easy)
    assert _same(pipe.result(t6), added[1]) and _same(pipe.result(t7), restored)
    t8 = pipe.submit(batch)
    with pytest.raises(m.MdirError, match="pending"):
        pipe.compact()
    pipe.result(t8)
    pipe.remove(new_ids.numpy())
    assert pipe.compact() == new_ids.numel()
    t9 = pipe.submit(batch)
    assert _same(pipe.result(t9), _np(g.search(batch, k=100, **p)))
    assert _same(pipe.result(pipe.submit(easy)), _np(g.search(easy, k=100, **p)))
    assert pipe.n_recovered == 6                                           # every hard ticket: t0, t2, t3, t5, t8, t9
