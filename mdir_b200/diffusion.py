"""Diffusion re-ranking on a mutual kNN graph of the database (Iscen, Tolias, Avrithis, Furon, Chum, CVPR 2017).

NOT in the reference (parity unpinned, like qe.py): the semantics are restated in tests/diffusion_reference.py:diffusion_graph
/ diffusion_search.  The graph is built once per index from the certified fp32 top-(k+1) of every row; a query's
certified fp32 shortlist L is re-ranked by f, the truncated CG solution of (I - alpha S_LL) f = y, where y holds the
query's top k_q scores raised to gamma.  The graph kernels and the per-query solve are mdir_b200/csrc/diffusion.cu."""
import math

import torch

from . import _lib
from .qe import DBA_BLOCK
from .search import Index, ShardedIndex, WIDE_Q, _as_dev_f32

MAX_K = 255          # neighbours per database row
MAX_TRUNC = 2048     # shortlist rows per query the solve kernel holds in shared memory


def check_graph_params(k, gamma):
    """MdirError unless 1 <= k <= 255 and gamma is finite and > 0."""
    if not 1 <= int(k) <= MAX_K:
        raise _lib.MdirError("diffusion needs 1 <= k <= %d neighbours per row (got %d)" % (MAX_K, int(k)))
    if not (math.isfinite(float(gamma)) and float(gamma) > 0):
        raise _lib.MdirError("diffusion needs a finite gamma > 0 (got %r)" % (gamma,))


def check_search_params(k, trunc, k_q, alpha, iters, rtol):
    """MdirError unless 1 <= k <= trunc <= 2048, 1 <= k_q <= trunc, 0 < alpha < 1, 1 <= iters <= 1000 and rtol >= 0."""
    k, trunc, k_q, iters = int(k), int(trunc), int(k_q), int(iters)
    if not 1 <= k <= trunc <= MAX_TRUNC:
        raise _lib.MdirError("diffusion needs 1 <= k <= trunc <= %d (got k=%d, trunc=%d)" % (MAX_TRUNC, k, trunc))
    if not 1 <= k_q <= trunc:
        raise _lib.MdirError("diffusion needs 1 <= k_q <= trunc (got k_q=%d, trunc=%d)" % (k_q, trunc))
    if not 0.0 < float(alpha) < 1.0:
        raise _lib.MdirError("diffusion needs 0 < alpha < 1 (got %r)" % (alpha,))
    if not 1 <= iters <= 1000:
        raise _lib.MdirError("diffusion needs 1 <= iters <= 1000 (got %d)" % iters)
    if not float(rtol) >= 0.0:
        raise _lib.MdirError("diffusion needs rtol >= 0 (got %r)" % (rtol,))


class Diffusion:
    """Diffusion search over a single-GPU Index.

        g = Diffusion(index, k=50, gamma=3.0)      # the graph: one wide search pass per 1,024 rows
        f, ids = g.search(q, k=100, trunc=1000, k_q=10, alpha=0.99, iters=20, rtol=1e-6)

    The index needs the fp32 master copy and no removed rows among its used slots (call compact() first; a free
    capacity tail is fine).  A later remove / restore / add / compact makes the graph stale: search() then raises
    until a new Diffusion is built."""

    def __init__(self, index, k=50, gamma=3.0):
        check_graph_params(k, gamma)
        if isinstance(index, ShardedIndex) or not isinstance(index, Index):
            raise _lib.MdirError("Diffusion needs a single-GPU Index (a ShardedIndex is not supported)")
        if index.db32 is None:
            raise _lib.MdirError("Diffusion needs the fp32 master copy (keep_fp32=True)")
        n_used = index._n_used
        if not index._live_host[:n_used].all():
            raise _lib.MdirError("Diffusion needs an index without removed rows (%d of %d used slots live): call compact() first"
                                 % (int(index._live_host[:n_used].sum()), n_used))
        self.index, self.k, self.gamma = index, int(k), float(gamma)
        self._version = index._mutations
        self._status = None
        dev = index.device
        with torch.cuda.device(dev):
            knn_i = torch.empty((n_used, self.k + 1), dtype=torch.int32, device=dev)
            knn_s = torch.empty((n_used, self.k + 1), dtype=torch.float32, device=dev)
            for r0 in range(0, n_used, DBA_BLOCK):
                r1 = min(r0 + DBA_BLOCK, n_used)
                s, i = index.search(index.db32[r0:r1], self.k + 1, precision="fp32", block_q=WIDE_Q)
                knn_s[r0:r1] = s
                knn_i[r0:r1] = i
            self.nbr = torch.empty((n_used, self.k), dtype=torch.int32, device=dev)
            self.S = torch.empty((n_used, self.k), dtype=torch.float32, device=dev)
            self.deg = torch.empty((n_used,), dtype=torch.float32, device=dev)
            lib = _lib.lib()
            _lib.check(lib.mdir_diffusion_graph(_lib.ptr(knn_i), _lib.ptr(knn_s), n_used, self.k, _lib.ptr(index.slot_id), self.gamma,
                                                _lib.ptr(self.nbr), _lib.ptr(self.S), _lib.ptr(self.deg), _lib.stream()), "mdir_diffusion_graph")
            _lib.check(lib.mdir_diffusion_normalize(_lib.ptr(self.nbr), _lib.ptr(self.S), _lib.ptr(self.deg), n_used, self.k, _lib.ptr(self.S),
                                                    _lib.stream()), "mdir_diffusion_normalize")

    def graph(self):
        """(nbr (n_used, k) int32 neighbour slots, mutual ones first and -1 padding; S (n_used, k) fp32 normalised
        weights aligned with nbr; deg (n_used,) fp32 degrees), on the device."""
        return self.nbr, self.S, self.deg

    def status(self):
        """Per-query status words of the last search()'s shortlist search (Index.status(): 0 = exact and certified)."""
        return self._status

    def search(self, q, k=100, trunc=1000, k_q=10, alpha=0.99, iters=20, rtol=1e-6):
        """q: (N_q, D) fp32 (host or device).  Returns (f (N_q, k) fp32, ids (N_q, k) int32) on the device: the shortlist
        L = index.search(q, trunc, precision="fp32") ranked by (f desc, position in L asc), f the CG solution of
        (I - alpha S_LL) f = y with y_u = max(s_u, 0)^gamma on the first k_q rows of L; -inf / -1 padding past |L|."""
        check_search_params(k, trunc, k_q, alpha, iters, rtol)
        index = self.index
        if index._mutations != self._version:
            raise _lib.MdirError("the index was mutated (remove / restore / add / compact) after the diffusion graph was built: "
                                 "build a new Diffusion")
        k, trunc = int(k), int(trunc)
        dev = index.device
        with torch.cuda.device(dev):
            q32 = _as_dev_f32(q, dev)
            n_q = q32.shape[0]
            f = torch.empty((n_q, k), dtype=torch.float32, device=dev)
            out = torch.empty((n_q, k), dtype=torch.int32, device=dev)
            if n_q == 0:
                self._status = torch.empty((0,), dtype=torch.int32, device=dev)
                return f, out
            s, ids = index.search(q32, trunc, precision="fp32", check=True)
            self._status = index.status()[:n_q].clone()
            lib = _lib.lib()
            ws_bytes = lib.mdir_diffusion_solve_workspace_bytes(n_q, trunc, self.k)
            ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
            _lib.check(lib.mdir_diffusion_solve(_lib.ptr(ids), _lib.ptr(s), n_q, trunc, _lib.ptr(index.slot_id), self.nbr.shape[0],
                                                _lib.ptr(self.nbr), _lib.ptr(self.S), self.k, int(k_q), self.gamma, float(alpha),
                                                int(iters), float(rtol), k, _lib.ptr(ws), ws_bytes, _lib.ptr(f), _lib.ptr(out),
                                                _lib.stream()), "mdir_diffusion_solve")
            return f, out
