"""CPU checks of diffusion re-ranking: the reference CG of tests/diffusion_reference.py against scipy and
np.linalg.solve, its mutual kNN graph against a loop-by-loop restatement of its definition (symmetry, weights from the lower slot, self-dropping among
duplicates), and the parameter refusals of mdir_b200.Diffusion, which need no GPU."""
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.sparse.linalg import cg as scipy_cg

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import diffusion_reference as dref  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def knn_lists(X, k1):
    """Exact top-k1 of every row against X by (score desc, id asc): ids and fp32 scores."""
    sc = (X.astype(np.float64) @ X.T.astype(np.float64)).astype(np.float32)
    idx = np.lexsort((np.broadcast_to(np.arange(X.shape[0]), sc.shape), -sc), axis=1)[:, :k1]
    return idx, np.take_along_axis(sc, idx, 1)


def unit_rows(n, D, seed):
    rs = np.random.RandomState(seed)
    X = rs.randn(n, D).astype(np.float32)
    return X / np.linalg.norm(X, axis=1, keepdims=True)


def spd_system(n, alpha, seed):
    """I - alpha S for the normalised graph of random unit rows (k = 8)."""
    X = unit_rows(n, 16, seed)
    ids, s = knn_lists(X, 9)
    nbr, S, _ = dref.diffusion_graph(ids, s, 8, 3.0)
    A = np.eye(n)
    for i in range(n):
        for e in range(8):
            if nbr[i, e] >= 0:
                A[i, nbr[i, e]] -= alpha * np.float64(S[i, e])
    return A


@pytest.mark.parametrize("rtol,maxiter", [(1e-6, 20), (1e-2, 50), (1e-12, 3), (0.5, 10)])
def test_cg_equals_scipy(rtol, maxiter):
    A = spd_system(300, 0.99, 1)
    rs = np.random.RandomState(2)
    y = np.zeros(300)
    y[:10] = rs.rand(10) ** 3
    runs = []
    ref, _ = scipy_cg(A, y, rtol=rtol, atol=0.0, maxiter=maxiter, callback=lambda xk: runs.append(1))
    x, it = dref.diffusion_cg(A, y, rtol, maxiter)
    assert it == len(runs)                                  # the same stopping decision
    np.testing.assert_allclose(x, ref, rtol=1e-12, atol=1e-14 * np.abs(ref).max())


def test_cg_zero_rhs():
    A = spd_system(50, 0.5, 3)
    ref, info = scipy_cg(A, np.zeros(50), rtol=1e-6, atol=0.0, maxiter=20)
    x, it = dref.diffusion_cg(A, np.zeros(50), 1e-6, 20)
    assert it == 0 and info == 0 and not x.any() and not ref.any()


def test_cg_converges_to_solve():
    A = spd_system(400, 0.99, 4)
    y = np.zeros(400)
    y[:25] = np.random.RandomState(5).rand(25)
    x, it = dref.diffusion_cg(A, y, 1e-13, 1000)
    assert it < 1000
    np.testing.assert_allclose(x, np.linalg.solve(A, y), rtol=0, atol=1e-11 * np.abs(x).max())


def test_cg_exact_zero_residual_stops():
    # one row: x = y after one step and r = 0 exactly; rtol = 0 would make scipy divide 0 by 0
    x, it = dref.diffusion_cg(np.eye(1), np.array([0.5]), 0.0, 5)
    assert x[0] == 0.5 and it == 1


def graph_by_definition(ids, s, k, gamma):
    """Loop-by-loop restatement: N(i), mutual edges, w from the lower slot, deg in N(i) order, S."""
    n = ids.shape[0]
    N = []
    for i in range(n):
        lst = [(int(j), np.float32(v)) for j, v in zip(ids[i], s[i]) if j != -1]
        if any(j == i for j, _ in lst):
            lst = [(j, v) for j, v in lst if j != i]
        else:
            lst = lst[:k]
        N.append(lst)
    Nset = [{j for j, _ in lst} for lst in N]
    sc = [{j: v for j, v in lst} for lst in N]
    nbr, W = [], []
    for i in range(n):
        row = [(j, np.power(max(sc[min(i, j)][max(i, j)], np.float32(0)), np.float32(gamma))) for j, _ in N[i] if i in Nset[j]]
        nbr.append([j for j, _ in row])
        W.append([w for _, w in row])
    deg = np.zeros(n, np.float32)
    for i in range(n):
        for w in W[i]:
            deg[i] = np.float32(deg[i] + w)
    return nbr, W, deg


@pytest.mark.parametrize("dups", [False, True])
def test_graph_matches_definition_and_is_symmetric(dups):
    k, gamma = 10, 3.0
    X = unit_rows(400, 16, 6)
    if dups:
        X[200:260] = X[100:160]                           # 60 exact duplicate pairs
        X[300:315] = X[0]                                  # 16 copies of one row: more than k + 1 tie at the top
    ids, s = knn_lists(X, k + 1)
    nbr, S, deg = dref.diffusion_graph(ids, s, k, gamma)
    ref_nbr, ref_w, ref_deg = graph_by_definition(ids, s, k, gamma)
    assert np.array_equal(deg, ref_deg)
    edges = {}
    for i in range(400):
        m = len(ref_nbr[i])
        assert list(nbr[i, :m]) == ref_nbr[i] and (nbr[i, m:] == -1).all() and (S[i, m:] == 0).all()
        for e, j in enumerate(ref_nbr[i]):
            w = ref_w[i][e]
            want = w / (np.sqrt(ref_deg[i]) * np.sqrt(ref_deg[j])) if w > 0 else np.float32(0)
            assert S[i, e] == np.float32(want)
            edges[(i, j)] = S[i, e]
    for (i, j), v in edges.items():                        # symmetric edge set, bitwise symmetric S
        assert edges[(j, i)].tobytes() == v.tobytes()
    assert len(edges) > 400


def test_self_dropped_among_duplicates():
    k = 4
    X = unit_rows(50, 16, 7)
    X[10] = X[3]                                           # row 10 ranks row 3 first (equal score, lower id), itself second
    X[20:27] = X[5]                                        # rows 5, 20..26 tie: row 26's top 5 are 5, 20, 21, 22, 23
    ids, s = knn_lists(X, k + 1)
    assert ids[10, 0] == 3 and ids[10, 1] == 10 and 26 not in ids[26]
    nbr, _, _ = dref.diffusion_graph(ids, s, k, 3.0)
    assert 10 not in nbr[10] and 3 in nbr[10] and 10 in nbr[3]
    # row 26 is not in its own list: its last entry is dropped, so N(26) = 5, 20, 21, 22 -- and none of those lists
    # (each holds itself) reaches 26, so row 26 has no mutual neighbour
    assert (nbr[26] == -1).all()


def test_parameter_refusals_without_gpu():
    import mdir_b200
    from mdir_b200 import diffusion as dif
    from mdir_b200.search import Index, ShardedIndex
    E = mdir_b200.MdirError
    for k, gamma in [(0, 3.0), (256, 3.0), (10, 0.0), (10, -1.0), (10, float("inf")), (10, float("nan"))]:
        with pytest.raises(E):
            dif.check_graph_params(k, gamma)
    dif.check_graph_params(255, 0.5)
    bad = [dict(k=0), dict(k=1001), dict(trunc=2049, k=100), dict(k_q=0), dict(k_q=1001), dict(alpha=0.0), dict(alpha=1.0),
           dict(alpha=float("nan")), dict(iters=0), dict(iters=1001), dict(rtol=-1e-6), dict(rtol=float("nan"))]
    base = dict(k=100, trunc=1000, k_q=10, alpha=0.99, iters=20, rtol=1e-6)
    for b in bad:
        with pytest.raises(E):
            dif.check_search_params(**{**base, **b})
    dif.check_search_params(k=2048, trunc=2048, k_q=2048, alpha=0.5, iters=1000, rtol=0.0)
    with pytest.raises(E, match="ShardedIndex"):
        mdir_b200.Diffusion(ShardedIndex.__new__(ShardedIndex))
    idx = Index.__new__(Index)
    idx.db32 = None
    with pytest.raises(E, match="fp32 master"):
        mdir_b200.Diffusion(idx)
    idx.db32 = np.zeros((4, 8), np.float32)
    idx._n_used = 3
    idx._live_host = np.array([True, False, True, False])
    with pytest.raises(E, match="compact"):
        mdir_b200.Diffusion(idx)
    with pytest.raises(E):
        mdir_b200.Diffusion(idx, k=0)


def test_product_imports_neither_oracle_nor_scipy():
    code = "import sys, mdir_b200, mdir_b200.diffusion; bad = [m for m in sys.modules if m.split('.')[0] in ('oracle', 'scipy')]; " \
           "assert not bad, bad"
    subprocess.run([sys.executable, "-c", code], cwd=ROOT, check=True)
