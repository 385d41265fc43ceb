"""Reference restatement of diffusion re-ranking (Iscen, Tolias, Avrithis, Furon, Chum, CVPR 2017) for the tests of
mdir_b200.Diffusion.  Not in the reference implementation (parity unpinned, like alpha_qe / dba in oracle/oracle.py):
numpy only, fp64 where the definition leaves the precision open.  tests/test_diffusion_oracle.py checks it against
scipy's cg and np.linalg.solve; tests/test_gpu_diffusion.py checks the CUDA path against it."""
import numpy as np


def diffusion_graph(knn_ids, knn_s, k, gamma=3.0, slot_id=None):
    """Iscen et al. CVPR'17 diffusion: the mutual kNN graph of a database (not in the reference; parity unpinned).

    knn_ids / knn_s (n, k + 1): every row's exact fp32 top-(k+1) against the database, ordered by (score desc,
    id asc), as ids (-1 padding) and scores; row r is slot r, whose id is slot_id[r] (increasing; default r).
    N(i) = the list without i itself wherever it lands, or without its last entry when i is not in it.
    (i, j) is an edge iff j in N(i) and i in N(j); w_ij = max(s, 0)^gamma in fp32, s from the list of the lower
    slot of i and j (so w is symmetric bit for bit); d_i = the fp32 sum of w_ij in N(i)'s order;
    S_ij = w_ij / (sqrt(d_i) sqrt(d_j)) in fp32 (0 where w_ij = 0).
    Returns nbr (n, k) int32 (mutual neighbours' slots in N(i) order, then -1), S (n, k) fp32, deg (n,) fp32."""
    knn_ids = np.asarray(knn_ids, dtype=np.int64)
    knn_s = np.asarray(knn_s, dtype=np.float32)
    n = knn_ids.shape[0]
    slot_id = np.arange(n, dtype=np.int64) if slot_id is None else np.asarray(slot_id, dtype=np.int64)
    pos = np.clip(np.searchsorted(slot_id, knn_ids), 0, n - 1)
    slots = np.where((knn_ids != -1) & (slot_id[pos] == knn_ids), pos, -1)
    rows = np.arange(n)[:, None]
    is_self = slots == rows
    keep = ~is_self
    keep[~is_self.any(1), k] = False                          # i not in its own list: drop the last entry
    N = slots[keep].reshape(n, k)
    sN = knn_s[keep].reshape(n, k)
    Nj = np.where(N >= 0, N, 0)
    mutual = np.zeros((n, k), dtype=bool)
    t = np.zeros((n, k), dtype=np.int64)
    for r0 in range(0, n, 2048):                              # (rows, k, k): i at position t of N(j)
        back = (N[Nj[r0:r0 + 2048]] == rows[r0:r0 + 2048, :, None]) & (N[r0:r0 + 2048] >= 0)[:, :, None]
        mutual[r0:r0 + 2048] = back.any(2)
        t[r0:r0 + 2048] = back.argmax(2)
    s = np.where(rows < N, sN, sN[Nj, t])
    w = np.where(mutual, np.power(np.maximum(s, np.float32(0)), np.float32(gamma)), np.float32(0)).astype(np.float32)
    order = np.argsort(~mutual, axis=1, kind="stable")        # mutual ones first, in N(i) order
    nbr = np.where(np.take_along_axis(mutual, order, 1), np.take_along_axis(N, order, 1), -1).astype(np.int32)
    w = np.take_along_axis(w, order, 1)
    deg = np.zeros(n, dtype=np.float32)
    for e in range(k):                                        # fp32, in N(i)'s order
        deg += w[:, e]
    dj = deg[np.where(nbr >= 0, nbr, 0)]
    with np.errstate(divide="ignore", invalid="ignore"):
        S = np.where(w > 0, w / (np.sqrt(deg)[:, None] * np.sqrt(dj)), np.float32(0)).astype(np.float32)
    return nbr, S, deg


def diffusion_cg(A, b, rtol, maxiter):
    """scipy.sparse.linalg.cg(A, b, rtol=rtol, atol=0, maxiter=maxiter) from x0 = 0, in fp64: stop when
    ||r|| < rtol ||b|| (tested at the top of each iteration), zeros when b = 0.  One addition: stop when r is exactly
    0 (rtol = 0), where scipy goes on to divide 0 by 0.  A: a dense (n, n) matrix.  Returns (x, iterations run)."""
    A = np.asarray(A, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    x = np.zeros_like(b)
    atol = rtol * np.linalg.norm(b)
    if not b.any():
        return x, 0
    r = b.copy()
    p = None
    rho_prev = None
    for it in range(maxiter):
        rho = r @ r
        if np.sqrt(rho) < atol or rho == 0:
            return x, it
        p = r.copy() if it == 0 else p * (rho / rho_prev) + r
        q = A @ p
        a = rho / (p @ q)
        x += a * p
        r -= a * q
        rho_prev = rho
    return x, maxiter


def diffusion_search(L_ids, L_s, nbr, S, k_out, k_q=10, gamma=3.0, alpha=0.99, iters=20, rtol=1e-6, slot_id=None):
    """Diffusion re-ranking of shortlists (not in the reference; parity unpinned).  L_ids / L_s (n_q, trunc): each
    query's exact fp32 top-trunc ids (-1 padding after the |L| rows found) and scores; nbr / S: diffusion_graph.
    y_u = max(s_u, 0)^gamma for the first k_q positions of L, else 0; f = diffusion_cg(I - alpha S_LL, y) in fp64;
    L ranked by (f desc, position asc).  Returns (f (n_q, k_out) fp64, ids (n_q, k_out) int64, -inf / -1 padding,
    and the list of every query's full f over L)."""
    L_ids = np.asarray(L_ids, dtype=np.int64)
    L_s = np.asarray(L_s, dtype=np.float32)
    nbr = np.asarray(nbr)
    S = np.asarray(S, dtype=np.float32)
    n_q, trunc = L_ids.shape
    slot_id = np.arange(nbr.shape[0], dtype=np.int64) if slot_id is None else np.asarray(slot_id, dtype=np.int64)
    f_out = np.full((n_q, k_out), -np.inf)
    ids_out = np.full((n_q, k_out), -1, dtype=np.int64)
    fulls = []
    for q in range(n_q):
        n = int(np.argmax(L_ids[q] == -1)) if (L_ids[q] == -1).any() else trunc
        slots = np.searchsorted(slot_id, L_ids[q, :n])
        local = {int(s): u for u, s in enumerate(slots)}
        A = np.eye(n)
        for u, s in enumerate(slots):
            for e in range(nbr.shape[1]):
                j = int(nbr[s, e])
                if j < 0:
                    break
                v = local.get(j)
                if v is not None:
                    A[u, v] -= alpha * np.float64(S[s, e])
        y = np.zeros(n)
        m = min(k_q, n)
        y[:m] = np.power(np.maximum(L_s[q, :m].astype(np.float64), 0.0), gamma)
        f, _ = diffusion_cg(A, y, rtol, iters)
        order = np.lexsort((np.arange(n), -f))[:k_out]
        f_out[q, :order.size] = f[order]
        ids_out[q, :order.size] = L_ids[q, order]
        fulls.append(f)
    return f_out, ids_out, fulls
