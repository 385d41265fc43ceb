"""Diffusion.add / remove / restore / compact on the GPU: after every update the raw top-(k+1) lists equal a fresh
certified search of every live row bit for bit (ids and fp32 score bits), removed rows hold padding, and the graph and
search outputs equal those of a new Diffusion over the same index bit for bit (DESIGN 2.2e)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import diffusion_reference as dref  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N_DB, D, K = 20000, 128, 50


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def _unit(x):
    return x / x.norm(dim=1, keepdim=True)


def make_db(dist, n, dim, seed):
    """n unit rows: randn (with 81 exact copies of row 999), clusters (200 centres) or near_dup (8 groups of 200 rows
    around random directions)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    if dist == "randn":
        db = _unit(torch.randn((n, dim), device=DEV, generator=g))
        db[1000:1080] = db[999]
    elif dist == "clusters":
        cent = torch.randn((200, dim), device=DEV, generator=g)
        c = torch.randint(0, 200, (n,), device=DEV, generator=g)
        db = _unit(cent[c] + 0.7 * torch.randn((n, dim), device=DEV, generator=g))
    elif dist == "near_dup":
        db = _unit(torch.randn((n, dim), device=DEV, generator=g))
        pos = torch.randperm(n, device=DEV, generator=g)[:1600].view(8, 200)
        for j in range(8):
            d = _unit(torch.randn((1, dim), device=DEV, generator=g))
            db[pos[j]] = _unit(d + 0.484 * torch.randn((200, dim), device=DEV, generator=g) / dim ** 0.5)
    else:
        raise ValueError(dist)
    return db


def knn_lists(m, index, k):
    """The graph build's own search call: top-(k+1) of every used row, DBA_BLOCK rows per call, wide passes."""
    from mdir_b200.qe import DBA_BLOCK
    from mdir_b200.search import WIDE_Q
    ids, sc = [], []
    for r0 in range(0, index._n_used, DBA_BLOCK):
        s, i = index.search(index.db32[r0:min(r0 + DBA_BLOCK, index._n_used)], k + 1, precision="fp32", block_q=WIDE_Q)
        ids.append(i.cpu().numpy())
        sc.append(s.cpu().numpy())
    return np.concatenate(ids).astype(np.int64), np.concatenate(sc)


def check_lists(m, g):
    """Live slots: the raw list equals a fresh search bit for bit; removed slots: padding.  Returns the fresh lists."""
    index = g.index
    n = index._n_used
    ids, sc = knn_lists(m, index, g.k)
    live = index._live_host[:n]
    gi, gs = g.knn_i[:n].cpu().numpy().astype(np.int64), g.knn_s[:n].cpu().numpy()
    bad = np.flatnonzero(live & ((gi != ids).any(1) | (gs.view(np.uint32) != sc.view(np.uint32)).any(1)))
    assert bad.size == 0, "lists differ at slots %s" % bad[:10]
    assert (gi[~live] == -1).all() and np.isneginf(gs[~live]).all()
    ids[~live], sc[~live] = -1, -np.inf
    assert (g.knn_i[n:] == -1).all() and torch.isneginf(g.knn_s[n:]).all()
    return ids, sc


def gpu_graph(m, index, ids, sc, k, gamma=3.0):
    """mdir_diffusion_graph + mdir_diffusion_normalize run on host lists."""
    from mdir_b200 import _lib
    n = ids.shape[0]
    ki = torch.from_numpy(ids.astype(np.int32)).to(DEV)
    ks = torch.from_numpy(sc).to(DEV)
    nbr = torch.empty((n, k), dtype=torch.int32, device=DEV)
    S = torch.empty((n, k), dtype=torch.float32, device=DEV)
    deg = torch.empty((n,), dtype=torch.float32, device=DEV)
    lib = _lib.lib()
    _lib.check(lib.mdir_diffusion_graph(_lib.ptr(ki), _lib.ptr(ks), n, k, _lib.ptr(index.slot_id), gamma, _lib.ptr(nbr), _lib.ptr(S),
                                        _lib.ptr(deg), _lib.stream()))
    _lib.check(lib.mdir_diffusion_normalize(_lib.ptr(nbr), _lib.ptr(S), _lib.ptr(deg), n, k, _lib.ptr(S), _lib.stream()))
    return nbr, S, deg


def check_graph(m, g, ids, sc):
    """The graph equals the reference's on the fresh lists (edges exactly, S / deg to 1e-6) and the GPU kernels' on
    those lists bit for bit."""
    nbr, S, deg = g.graph()
    r_nbr, r_S, r_deg = dref.diffusion_graph(ids, sc, g.k, g.gamma, slot_id=g.index._ids)
    assert np.array_equal(nbr.cpu().numpy(), r_nbr)
    np.testing.assert_allclose(S.cpu().numpy(), r_S, rtol=1e-6, atol=0)
    np.testing.assert_allclose(deg.cpu().numpy(), r_deg, rtol=1e-6, atol=0)
    b_nbr, b_S, b_deg = gpu_graph(m, g.index, ids, sc, g.k, g.gamma)
    assert torch.equal(nbr, b_nbr) and torch.equal(S.view(torch.int32), b_S.view(torch.int32))
    assert torch.equal(deg.view(torch.int32), b_deg.view(torch.int32))


def check_rebuild(m, g, q=None):
    """graph() (and search() on q) equal those of a new Diffusion over the index, bit for bit."""
    fresh = m.Diffusion(g.index, k=g.k, gamma=g.gamma)
    for a, b in zip(g.graph(), fresh.graph()):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    if q is not None:
        f1, i1 = g.search(q, k=100, trunc=500)
        s1 = g.status().clone()
        f2, i2 = fresh.search(q, k=100, trunc=500)
        assert torch.equal(f1.view(torch.int32), f2.view(torch.int32)) and torch.equal(i1, i2)
        assert torch.equal(s1, fresh.status())


def batches(db, seed, sizes, dim):
    """New rows: noisy copies of random existing rows, with exact copies of existing rows in the 37-row batch and 60
    near-duplicates of row 123 (more than k + 1) in the 1,024-row batch."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    out = []
    for nb in sizes:
        src = torch.randint(0, db.shape[0], (nb,), device=DEV, generator=g)
        x = _unit(db[src] + 0.3 * torch.randn((nb, dim), device=DEV, generator=g) / dim ** 0.5)
        if nb == 37:
            x[:12] = db[5:17]                                             # exact duplicates: ties decided by id
        if nb == 1024:
            x[100:160] = _unit(db[123][None, :] + 0.01 * torch.randn((60, dim), device=DEV, generator=g) / dim ** 0.5)
        out.append(x)
    return out


@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
def test_add_matches_rebuild(m, dist):
    db = make_db(dist, N_DB, D, 31)
    sizes = [1, 37, 1024, 3000]
    index = m.Index(db, device=DEV, capacity=N_DB + sum(sizes))
    g = m.Diffusion(index, k=K, gamma=3.0)
    searched = 0
    for x in batches(db, 5, sizes, D):
        ids = g.add(x)
        assert ids.numel() == x.shape[0]
        searched += x.shape[0]
        assert g.update_stats["rows_searched"] == searched                # only the new rows were searched
        kid, ksc = check_lists(m, g)
        check_rebuild(m, g)
    check_graph(m, g, kid, ksc)
    q = _unit(db[:40] + 0.5 * torch.randn((40, D), device=DEV, generator=torch.Generator(device=DEV).manual_seed(2)) / D ** 0.5)
    check_rebuild(m, g, q)
    st = g.update_stats
    assert st["replaced"] > 0 and st["screen_passed"] >= st["rescored"] >= st["replaced"]


def test_add_2048(m):
    dim = 2048
    db = make_db("clusters", 8000, dim, 41)
    index = m.Index(db, device=DEV, capacity=8000 + 1061)
    g = m.Diffusion(index, k=K)
    for x in batches(db, 6, [37, 1024], dim):
        g.add(x)
    check_lists(m, g)
    check_rebuild(m, g, _unit(db[:16] + 0.01 * torch.randn((16, dim), device=DEV)))


def _holders(lists_ids, ids):
    """Rows whose list holds one of these ids."""
    return np.flatnonzero(np.isin(lists_ids, ids).any(1))


@pytest.mark.parametrize("which", ["random", "cluster", "neighbours"])
def test_remove_restore(m, which):
    db = make_db("clusters", N_DB, D, 51)
    index = m.Index(db, device=DEV)
    g = m.Diffusion(index, k=K)
    kid0, _ = knn_lists(m, index, K)
    if which == "random":
        gone = np.random.RandomState(1).choice(N_DB, 300, replace=False)
    elif which == "cluster":                                              # the 40 nearest rows of row 10 and their lists
        gone = np.unique(kid0[kid0[10, :40]].ravel())
    else:
        gone = kid0[77].copy()                                            # every neighbour of row 77, row 77 included
    A = np.setdiff1d(_holders(kid0, gone), gone)
    g.remove(gone)
    assert g.update_stats["rows_searched"] == A.size                      # only the rows that held a removed id
    kid, ksc = check_lists(m, g)
    check_graph(m, g, kid, ksc)
    nbr, _, deg = g.graph()
    assert (nbr[torch.from_numpy(gone).to(DEV)] == -1).all() and (deg[torch.from_numpy(gone).to(DEV)] == 0).all()
    g.restore(gone)
    assert g.update_stats["rows_searched"] == A.size + gone.size
    kid, ksc = check_lists(m, g)
    check_graph(m, g, kid, ksc)
    check_rebuild(m, g)


def test_mixed_sequence_then_compact(m):
    db = make_db("randn", N_DB, D, 61)
    index = m.Index(db[:15000], device=DEV, capacity=N_DB)
    g = m.Diffusion(index, k=K)
    rs = np.random.RandomState(7)
    removed, nxt = [], 15000
    for step in range(8):
        op = ["add", "remove", "restore", "compact"][step % 4]
        if op == "add":
            n_add = int(rs.randint(1, 600))
            g.add(db[nxt:nxt + n_add])
            nxt += n_add
        elif op == "remove":
            ids = rs.choice(index._ids[index._live_host[:index._n_used]], 400, replace=False)
            g.remove(ids)
            removed.append(ids)
        elif op == "restore":
            g.restore(removed[-1][:150])
        else:
            g.compact()
        check_lists(m, g)
    g.remove(rs.choice(index._ids, 500, replace=False))
    assert g.compact() > 0
    old_max = int(index._ids.max())
    ids = g.add(db[nxt:nxt + 700])                                        # into slots freed by compaction: new ids
    assert int(ids.min()) > old_max
    check_lists(m, g)
    q = _unit(db[:50] + 0.5 * torch.randn((50, D), device=DEV, generator=torch.Generator(device=DEV).manual_seed(3)) / D ** 0.5)
    check_rebuild(m, g, q)


def test_screen_overflow_rerun(m, monkeypatch):
    import mdir_b200.diffusion as dmod
    db = make_db("near_dup", N_DB, D, 71)
    index = m.Index(db, device=DEV, capacity=N_DB + 400)
    g = m.Diffusion(index, k=K)
    src = torch.arange(0, N_DB, 50, device=DEV)
    x = _unit(db[src] + 1e-3 * torch.randn((src.numel(), D), device=DEV) / D ** 0.5)      # near-duplicates of 400 rows
    monkeypatch.setattr(dmod, "MERGE_CAP", 2)
    g.add(x)
    st = g.update_stats
    assert st["screen_reruns"] > 0 and st["screen_passed"] > st["rescored"]
    assert st["rescored"] > st["replaced"] > 0                            # pairs within eps of T_i that did not enter
    check_lists(m, g)
    check_rebuild(m, g)


def test_edges(m):
    db = make_db("clusters", 3000, D, 81)
    # fewer than k + 1 live rows: every list has padding, every pair passes the screen
    index = m.Index(db[:30], device=DEV, capacity=60)
    g = m.Diffusion(index, k=K)
    g.add(db[30:45])
    check_lists(m, g)
    check_rebuild(m, g)
    g.add(db[45:60])                                                      # fills the last free slot exactly
    assert index._n_used == index.n
    check_lists(m, g)
    check_rebuild(m, g)
    # every row of one cluster removed
    index = m.Index(db, device=DEV)
    g = m.Diffusion(index, k=K)
    kid, _ = knn_lists(m, index, K)
    cl = np.unique(kid[kid[0]].ravel())
    g.remove(cl)
    kid, ksc = check_lists(m, g)
    check_graph(m, g, kid, ksc)
    g.compact()
    check_rebuild(m, g)


def test_still_refused(m):
    db = make_db("randn", 6000, D, 91)
    index = m.Index(db[:5000], device=DEV, capacity=5100)
    g = m.Diffusion(index, k=20)
    g.add(db[5000:5050])
    g.search(db[:4], k=50, trunc=200)
    index.remove([3])                                                     # on the index directly
    with pytest.raises(m.MdirError, match="mutated"):
        g.search(db[:4], k=50, trunc=200)
    with pytest.raises(m.MdirError, match="mutated"):
        g.add(db[5050:5060])
    g = m.Diffusion(m.Index(db[:5000], device=DEV, capacity=5010), k=20)
    with pytest.raises(m.MdirError, match="full"):
        g.add(db[5000:5020])
    with pytest.raises(m.MdirError, match="never filled"):
        g.restore([5005])
    g.search(db[:4], k=50, trunc=200)                                     # still usable
    check_lists(m, g)
    check_rebuild(m, g)
