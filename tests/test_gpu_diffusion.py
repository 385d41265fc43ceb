"""mdir_b200.Diffusion on the GPU against tests/diffusion_reference.py:diffusion_graph / diffusion_search (fp64 CG,
equal to scipy's cg: tests/test_diffusion_oracle.py).  Both sides start from the same certified index.search lists, so the graph is
compared exactly (edge sets) and to 1e-6 (S, deg), and the solve to 1e-5 of max |f|.  Determinism, ids after compact(),
the refusals after a mutation and the mAP gain on chain-shaped classes are checked too."""
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
F_TOL = 1e-5          # max |f - f_ref| / max |f_ref| (the kernel's CG against the oracle's)


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def _unit(x):
    return x / x.norm(dim=1, keepdim=True)


def build_case(dist, seed=11, n_q=8):
    """(db, q) unit rows on the device.  randn carries 81 exact copies of one row (the copies past the first k + 1 are
    not in their own lists: isolated nodes), and its first query sits on that row."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    if dist == "randn":
        db = _unit(torch.randn((N_DB, D), device=DEV, generator=g))
        db[1000:1080] = db[999]
    elif dist == "clusters":
        cent = torch.randn((200, D), device=DEV, generator=g)
        c = torch.randint(0, 200, (N_DB,), device=DEV, generator=g)
        db = _unit(cent[c] + 0.7 * torch.randn((N_DB, D), device=DEV, generator=g))
    elif dist == "near_dup":
        db = _unit(torch.randn((N_DB, D), device=DEV, generator=g))
        q = _unit(torch.randn((n_q, D), device=DEV, generator=g))
        pos = torch.randperm(N_DB, device=DEV, generator=g)[:n_q * 200].view(n_q, 200)
        for j in range(n_q):                  # 200 near-duplicates per query
            nz = torch.randn((200, D), device=DEV, generator=g)
            nz = nz - (nz @ q[j])[:, None] * q[j][None, :]
            db[pos[j]] = _unit(q[j][None, :] + 0.484 * nz / D ** 0.5)
        return db, q
    else:
        raise ValueError(dist)
    src = torch.randperm(N_DB, device=DEV, generator=g)[:n_q]
    if dist == "randn":
        src[0] = 999
    q = _unit(db[src] + 0.5 * torch.randn((n_q, D), device=DEV, generator=g) / D ** 0.5)
    return db, q


_CASES = {}


def case(m, dist):
    """(index, Diffusion(k=50), q, knn ids, knn scores), built once per module."""
    if dist not in _CASES:
        db, q = build_case(dist)
        index = m.Index(db, device=DEV)
        g = m.Diffusion(index, k=K, gamma=3.0)
        ids, sc = knn_lists(m, index, K)
        _CASES[dist] = (index, g, q, ids, sc)
    return _CASES[dist]


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


def check_solve(f, ids, L_ids, ref_f_full, k_out):
    """f / ids of the GPU against the fp64 solve on the same L: |f - f_ref| <= F_TOL max |f_ref| at every returned row,
    and the ranking equal to the oracle's except between rows whose reference f differ by less than that bound."""
    f, ids = f.cpu().numpy(), ids.cpu().numpy()
    for qi in range(f.shape[0]):
        ref = ref_f_full[qi]
        n = ref.size
        bound = F_TOL * max(np.abs(ref).max(), np.finfo(np.float32).tiny)
        pos_of = {int(v): u for u, v in enumerate(L_ids[qi, :n])}
        m = min(k_out, n)
        assert (ids[qi, m:] == -1).all() and np.isneginf(f[qi, m:]).all()
        got_pos = np.array([pos_of[int(v)] for v in ids[qi, :m]])
        assert np.unique(got_pos).size == m
        assert np.abs(f[qi, :m] - ref[got_pos]).max(initial=0) <= bound, qi
        want_pos = np.lexsort((np.arange(n), -ref))[:m]
        diff = got_pos != want_pos
        assert np.all(np.abs(ref[got_pos[diff]] - ref[want_pos[diff]]) <= bound), qi


@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
def test_graph_matches_oracle(m, dist):
    index, g, _, ids, sc = case(m, dist)
    nbr, S, deg = (t.cpu().numpy() for t in g.graph())
    r_nbr, r_S, r_deg = dref.diffusion_graph(ids, sc, K, 3.0)
    assert np.array_equal(nbr, r_nbr)                                     # the same edges, in the same order
    np.testing.assert_allclose(S, r_S, rtol=1e-6, atol=0)
    np.testing.assert_allclose(deg, r_deg, rtol=1e-6, atol=0)
    ii, ee = np.nonzero(nbr >= 0)
    jj = nbr[ii, ee]
    back = np.argmax(nbr[jj] == ii[:, None], axis=1)
    assert (nbr[jj, back] == ii).all()
    assert np.array_equal(S[ii, ee].view(np.uint32), S[jj, back].view(np.uint32))   # bitwise symmetric
    if dist == "randn":
        assert ((nbr[1000:1080] == -1).all(1)).sum() >= 20 and (deg[1000:1080] == 0).sum() >= 20   # isolated copies


SOLVE = [(t, kq) for t in (1, 17, 1000, 2048) for kq in sorted({1, 10, t}) if kq <= t]


@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
@pytest.mark.parametrize("trunc,k_q", SOLVE)
def test_solve_matches_cg(m, dist, trunc, k_q):
    index, g, q, _, _ = case(m, dist)
    k_out = trunc if trunc <= 17 else 100                                 # k = trunc on the short lists
    f, ids = g.search(q, k=k_out, trunc=trunc, k_q=k_q, alpha=0.99, iters=20, rtol=1e-6)
    s, L = index.search(q, trunc, precision="fp32")
    assert torch.equal(g.status(), index.status()[:q.shape[0]])
    nbr, S, _ = g.graph()
    L = L.cpu().numpy().astype(np.int64)
    _, _, fulls = dref.diffusion_search(L, s.cpu().numpy(), nbr.cpu().numpy(), S.cpu().numpy(), k_out, k_q=k_q, gamma=3.0,
                                          alpha=0.99, iters=20, rtol=1e-6)
    check_solve(f, ids, L, fulls, k_out)


def test_zero_rhs_keeps_shortlist_order(m):
    # every row has a first coordinate in [0.5, 0.7] and the query is -e0: all scores are negative, so y = 0 and f = 0
    g0 = torch.Generator(device=DEV).manual_seed(3)
    db = torch.randn((3000, 64), device=DEV, generator=g0)
    db[:, 0] = 0.0
    x0 = 0.5 + 0.2 * torch.rand((3000,), device=DEV, generator=g0)
    db = _unit(db) * torch.sqrt(1 - x0 * x0)[:, None]
    db[:, 0] = x0
    q = torch.zeros((3, 64), device=DEV)
    q[:, 0] = -1.0
    index = m.Index(db, device=DEV)
    g = m.Diffusion(index, k=20)
    f, ids = g.search(q, k=50, trunc=300, k_q=10)
    _, L = index.search(q, 300, precision="fp32")
    assert (f == 0).all() and torch.equal(ids, L[:, :50])


def test_fewer_live_rows_than_trunc(m):
    db, q = build_case("clusters", seed=5)
    index = m.Index(db[:600], device=DEV, capacity=1000)                  # 600 live rows, a free tail of 400
    g = m.Diffusion(index, k=10)
    f, ids = g.search(q, k=1000, trunc=1000, k_q=10)
    s, L = index.search(q, 1000, precision="fp32")
    nbr, S, _ = g.graph()
    L = L.cpu().numpy().astype(np.int64)
    assert (L[:, 600:] == -1).all() and (L[:, :600] >= 0).all()
    _, _, fulls = dref.diffusion_search(L, s.cpu().numpy(), nbr.cpu().numpy(), S.cpu().numpy(), 1000, k_q=10)
    check_solve(f, ids, L, fulls, 1000)


def test_deterministic_and_batch_invariant(m):
    index, g, _, _, _ = case(m, "clusters")
    g0 = torch.Generator(device=DEV).manual_seed(21)
    src = torch.randint(0, N_DB, (200,), device=DEV, generator=g0)
    q = _unit(index.db32[src] + 0.5 * torch.randn((200, D), device=DEV, generator=g0) / D ** 0.5)   # 200 > 128: two scan blocks
    f1, i1 = g.search(q)
    f2, i2 = g.search(q)
    assert torch.equal(f1, f2) and torch.equal(i1, i2)
    for j in (0, 137, 199):
        fa, ia = g.search(q[j:j + 1])
        assert torch.equal(fa[0], f1[j]) and torch.equal(ia[0], i1[j]), j
    fb, ib = g.search(q[100:190])                                         # another batch composition
    assert torch.equal(fb, f1[100:190]) and torch.equal(ib, i1[100:190])


def test_ids_after_compact(m):
    db, q = build_case("clusters", seed=7)
    a = m.Index(db.clone(), device=DEV)                                  # compact() rewrites the master copy in place
    gone = np.random.RandomState(0).choice(N_DB, 3000, replace=False)
    a.remove(gone)
    a.compact()
    ga = m.Diffusion(a, k=K)
    live = np.setdiff1d(np.arange(N_DB), gone)
    b = m.Index(db[torch.from_numpy(live).to(DEV)], device=DEV)
    gb = m.Diffusion(b, k=K)
    fa, ia = ga.search(q)
    fb, ib = gb.search(q)
    assert torch.equal(fa, fb)
    assert np.array_equal(ia.cpu().numpy(), live[ib.cpu().numpy()])


def test_mutation_after_build_refused(m):
    db, q = build_case("randn", seed=9)
    index = m.Index(db[:5000], device=DEV, capacity=6000)
    g = m.Diffusion(index, k=20)
    g.search(q, k=50, trunc=200)
    index.remove([5])
    with pytest.raises(m.MdirError, match="mutated"):
        g.search(q, k=50, trunc=200)
    index.restore([5])                                                    # back to the same rows, but still a mutation
    with pytest.raises(m.MdirError, match="mutated"):
        g.search(q, k=50, trunc=200)
    for mutate in (lambda: index.add(db[5000:5010]), lambda: (index.remove([7]), index.compact())):
        g = m.Diffusion(index, k=20)                                      # a rebuild works
        g.search(q, k=50, trunc=200)
        mutate()
        with pytest.raises(m.MdirError, match="mutated"):
            g.search(q, k=50, trunc=200)
    g = m.Diffusion(index, k=20)
    g.search(q, k=50, trunc=200)
    index.remove([8])
    with pytest.raises(m.MdirError, match="compact"):
        m.Diffusion(index, k=20)


def chains(n_cls=100, per=100, dim=64, step=0.2, qnoise=0.3, seed=0):
    """n_cls classes, each a random walk of `per` unit vectors; one query per class near a random point of its walk."""
    rs = np.random.RandomState(seed)
    X = np.empty((n_cls * per, dim), np.float32)
    for c in range(n_cls):
        x = rs.randn(dim)
        x /= np.linalg.norm(x)
        for t in range(per):
            X[c * per + t] = x
            x = x + step * rs.randn(dim) / np.sqrt(dim)
            x /= np.linalg.norm(x)
    qi = np.arange(n_cls) * per + rs.randint(0, per, n_cls)
    Q = X[qi] + qnoise * rs.randn(n_cls, dim).astype(np.float32) / np.sqrt(dim)
    Q /= np.linalg.norm(Q, axis=1, keepdims=True)
    return X, Q.astype(np.float32), np.repeat(np.arange(n_cls), per)


def map_at(ids, lab, k=100):
    """Mean over queries (query c belongs to class c) of AP over the top k, normalised by min(class size, k)."""
    aps = []
    for c, row in enumerate(ids):
        rel = lab[row[:k]] == c
        aps.append((rel * np.cumsum(rel) / np.arange(1, k + 1)).sum() / min(k, int((lab == c).sum())))
    return float(np.mean(aps))


def test_map_on_chains(m):
    X, Q, lab = chains()
    index = m.Index(X, device=DEV)
    g = m.Diffusion(index, k=30, gamma=3.0)
    f, ids = g.search(Q, k=100, trunc=500, k_q=10, alpha=0.99, iters=20, rtol=1e-6)
    s, L = index.search(Q, 500, precision="fp32")
    kid, ksc = knn_lists(m, index, 30)
    nbr, S, _ = dref.diffusion_graph(kid, ksc, 30, 3.0)
    _, ref_ids, _ = dref.diffusion_search(L.cpu().numpy(), s.cpu().numpy(), nbr, S, 100, k_q=10, gamma=3.0, alpha=0.99,
                                            iters=20, rtol=1e-6)
    m_gpu, m_ref, m_plain = map_at(ids.cpu().numpy(), lab), map_at(ref_ids, lab), map_at(L.cpu().numpy(), lab)
    print("chain mAP@100: plain %.4f, diffusion %.4f (oracle %.4f)" % (m_plain, m_gpu, m_ref))
    assert abs(m_gpu - m_ref) <= 0.005
    assert m_gpu >= m_plain + 0.03
