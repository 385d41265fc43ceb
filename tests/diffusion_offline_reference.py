"""Reference restatement of offline diffusion (Yang, Hinami, Matsui, Ly, Satoh, AAAI 2019: diffusion decoupled into
online and offline processing) for the tests of mdir_b200.DiffusionTable.  Not in the reference implementation (parity
unpinned): numpy only, fp64 where the definition leaves the precision open, built on diffusion_reference.diffusion_search
with k_q = 1.  tests/test_diffusion_offline_oracle.py checks it against dense solves combined by linearity;
tests/test_gpu_diffusion_offline.py checks the CUDA path against it."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from diffusion_reference import diffusion_search  # noqa: E402


def offline_table(L_ids, L_s, nbr, S, width, gamma=3.0, alpha=0.99, iters=20, rtol=1e-6, slot_id=None):
    """Offline diffusion's table (Yang et al. AAAI 2019's decoupling; not in the reference, parity unpinned).  L_ids /
    L_s (n, trunc): row r's own exact fp32 top-trunc as a query (row r = slot r).  Row r of the table is diffusion_search
    of that shortlist with k_q = 1: the right-hand side seeded on the shortlist's first entry, which is the row itself
    or an exact duplicate with a lower id (both rows then get the same table row).  Returns (ids (n, width) int64, f
    (n, width) fp64), -1 / -inf padding."""
    f, ids, _ = diffusion_search(L_ids, L_s, nbr, S, width, k_q=1, gamma=gamma, alpha=alpha, iters=iters, rtol=rtol, slot_id=slot_id)
    return ids, f


def offline_search(table_ids, table_f, L_ids, L_s, k, gamma=3.0, slot_id=None):
    """Offline diffusion of queries from a table (offline_table's, or any with that layout; row r = slot r, whose id is
    slot_id[r]).  L_ids / L_s (n_q, k_q): each query's exact fp32 top-k_q (-1 padding).  w_u = max(s_u, 0)^gamma in
    fp64; for every id j in the union of the table rows of L's rows, f_j = sum over u ascending of w_u * F[slot(L_u)][j]
    in fp64; padding entries of L and of the table are skipped.  The top k by (fp32(f) desc, id asc).  Returns (f
    (n_q, k) fp64, ids (n_q, k) int64, -inf / -1 padding past the union, and every query's full {id: f} dict)."""
    table_ids = np.asarray(table_ids, dtype=np.int64)
    table_f = np.asarray(table_f, dtype=np.float64)
    L_ids = np.asarray(L_ids, dtype=np.int64)
    L_s = np.asarray(L_s, dtype=np.float32)
    slot_id = np.arange(table_ids.shape[0], dtype=np.int64) if slot_id is None else np.asarray(slot_id, dtype=np.int64)
    n_q = L_ids.shape[0]
    f_out = np.full((n_q, k), -np.inf)
    ids_out = np.full((n_q, k), -1, dtype=np.int64)
    fulls = []
    for q in range(n_q):
        acc = {}
        for u in range(L_ids.shape[1]):
            if L_ids[q, u] == -1:
                continue
            s = int(np.searchsorted(slot_id, L_ids[q, u]))
            w = np.power(max(np.float64(L_s[q, u]), 0.0), np.float64(gamma))
            for j, v in zip(table_ids[s], table_f[s]):
                if j != -1:
                    acc[int(j)] = acc.get(int(j), 0.0) + w * v
        ids = np.fromiter(acc.keys(), dtype=np.int64, count=len(acc))
        f = np.fromiter(acc.values(), dtype=np.float64, count=len(acc))
        order = np.lexsort((ids, -f.astype(np.float32)))[:k]
        f_out[q, :order.size] = f[order]
        ids_out[q, :order.size] = ids[order]
        fulls.append(acc)
    return f_out, ids_out, fulls
