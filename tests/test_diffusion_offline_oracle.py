"""CPU checks of offline diffusion: the restatement of tests/diffusion_offline_reference.py (offline_table /
offline_search) against an independent path, the dense solve of every table row's system combined by linearity; its
ordering and padding on a hand-made table; and the parameter refusals of mdir_b200.DiffusionTable, which need no GPU."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import diffusion_offline_reference as oref  # noqa: E402
import diffusion_reference as dref  # noqa: E402


def sorted_lists(X, Y, k):
    """Exact top-k of every row of Y against the rows of X by (score desc, id asc): ids and fp32 scores."""
    sc = (Y.astype(np.float64) @ X.T.astype(np.float64)).astype(np.float32)
    idx = np.lexsort((np.broadcast_to(np.arange(X.shape[0]), sc.shape), -sc), axis=1)[:, :k]
    return idx, np.take_along_axis(sc, idx, 1)


def unit_rows(n, D, seed):
    rs = np.random.RandomState(seed)
    X = rs.randn(n, D).astype(np.float32)
    return X / np.linalg.norm(X, axis=1, keepdims=True)


def test_offline_search_is_linear_in_the_seeds():
    n, k, gamma, alpha, k_q = 300, 10, 3.0, 0.99, 10
    X = unit_rows(n, 16, 1)
    X[200] = X[100]                                        # an exact duplicate: row 200's shortlist starts with row 100
    kid, ksc = sorted_lists(X, X, k + 1)
    nbr, S, _ = dref.diffusion_graph(kid, ksc, k, gamma)
    L_all, s_all = sorted_lists(X, X, n)                   # trunc = n: every row's shortlist holds all rows
    assert L_all[200, 0] == 100 and L_all[100, 0] == 100
    tab_ids, tab_f = oref.offline_table(L_all, s_all, nbr, S, n, gamma=gamma, alpha=alpha, iters=n, rtol=0.0)
    assert np.array_equal(tab_ids[200], tab_ids[100]) and np.array_equal(tab_f[200], tab_f[100])
    assert (tab_ids >= 0).all() and np.isfinite(tab_f).all()
    A = np.eye(n)
    for i in range(n):
        for e in range(k):
            if nbr[i, e] >= 0:
                A[i, nbr[i, e]] -= alpha * np.float64(S[i, e])
    Q = unit_rows(6, 16, 2)
    Q[0] = X[200]                                          # a query on the duplicate pair
    L_q, s_q = sorted_lists(X, Q, k_q)
    f, ids, fulls = oref.offline_search(tab_ids, tab_f, L_q, s_q, n, gamma=gamma)
    for qi in range(Q.shape[0]):
        ref = np.zeros(n)
        for u in range(k_q):
            j = L_q[qi, u]
            y = np.zeros(n)
            y[L_all[j, 0]] = np.power(max(np.float64(s_all[j, 0]), 0.0), gamma)
            ref += np.power(max(np.float64(s_q[qi, u]), 0.0), gamma) * np.linalg.solve(A, y)
        got = fulls[qi]
        assert sorted(got) == list(range(n))
        err = max(abs(got[j] - ref[j]) for j in range(n))
        assert err <= 1e-9 * np.abs(ref).max(), (qi, err)
        want = np.lexsort((np.arange(n), -ref.astype(np.float32)))
        assert np.array_equal(ids[qi], want) or np.abs(ref[ids[qi]] - ref[want]).max() <= 1e-9 * np.abs(ref).max()


def test_offline_search_union_order_and_padding():
    # slots 0..3 with ids 10, 20, 30, 40; width 3
    tab_ids = np.array([[10, 20, -1], [20, 30, 40], [30, -1, -1], [40, 10, 30]])
    tab_f = np.array([[1.0, 0.5, -np.inf], [2.0, 0.25, 0.25], [1.0, -np.inf, -np.inf], [4.0, 0.5, 0.5]], np.float32)
    slot_id = np.array([10, 20, 30, 40])
    L_ids = np.array([[10, 20], [30, -1], [-1, -1]])
    L_s = np.array([[1.0, 2 ** (1 / 3)], [-0.5, -np.inf], [-np.inf, -np.inf]], np.float32)
    f, ids, fulls = oref.offline_search(tab_ids, tab_f, L_ids, L_s, 5, gamma=3.0, slot_id=slot_id)
    w1 = np.power(np.float64(np.float32(2 ** (1 / 3))), 3.0)
    # query 0: 10 -> 1, 20 -> 0.5 + 2 w1, 30 -> 0.25 w1, 40 -> 0.25 w1 (a tie: the lower id first); no fifth id
    assert list(ids[0]) == [20, 10, 30, 40, -1]
    np.testing.assert_allclose(f[0, :4], [0.5 + 2 * w1, 1.0, 0.25 * w1, 0.25 * w1], rtol=1e-15)
    assert np.isneginf(f[0, 4])
    # query 1: a negative score gives w = 0, yet its table row's ids stay in the union (with f = 0)
    assert list(ids[1]) == [30, -1, -1, -1, -1] and f[1, 0] == 0.0
    assert list(ids[2]) == [-1] * 5 and np.isneginf(f[2]).all() and fulls[2] == {}


def test_offline_parameter_refusals_without_gpu():
    import mdir_b200
    from mdir_b200 import diffusion as dif
    from mdir_b200.search import ShardedIndex
    E = mdir_b200.MdirError
    base = dict(width=100, trunc=1000, alpha=0.99, iters=20, rtol=1e-6)
    for b in [dict(width=0), dict(width=1025, trunc=2048), dict(width=200, trunc=100), dict(trunc=2049), dict(alpha=1.0),
              dict(iters=0), dict(rtol=-1.0)]:
        with pytest.raises(E):
            dif.check_offline_params(**{**base, **b})
    dif.check_offline_params(width=1024, trunc=2048, alpha=0.5, iters=1000, rtol=0.0)
    for k, k_q, width in [(100, 0, 100), (100, 129, 10), (100, 82, 100), (0, 10, 100), (8193, 10, 100)]:
        with pytest.raises(E):
            dif.check_combine_params(k, k_q, width)
    dif.check_combine_params(8192, 8, 1024)
    dif.check_combine_params(1, 128, 64)
    g = dif.Diffusion.__new__(dif.Diffusion)
    g.index = ShardedIndex.__new__(ShardedIndex)
    with pytest.raises(E, match="ShardedIndex"):
        g.offline()
    with pytest.raises(E, match="width"):
        g.offline(width=0)
