"""Diffusion re-ranking at the R1M shape (1,001,001 x 2048 unit randn rows, k = 50, 70 queries, trunc = 1000, one GPU).

  * build  -- Diffusion(index, k=50): host clock around the constructor plus a device synchronise (the top-51 of every
              row in wide search passes of 1,024 rows, then mdir_diffusion_graph + _normalize).  The index's one-time
              certificate pass runs in a search before it, so it is not counted.  The search passes are then timed
              again alone.
  * search -- the shortlist search alone, index.search(q, 1000, precision="fp32"): CUDA events, median over REPS.
  * solve  -- mdir_diffusion_solve alone on that shortlist (k_q = 10, alpha = 0.99, iters = 20, rtol = 1e-6): CUDA events,
              median over REPS.
  * step   -- Diffusion.search(q) end to end: host clock around the call plus a device synchronise, median over REPS.

    python tools/time_diffusion.py
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mdir_b200  # noqa: E402
from mdir_b200 import _lib  # noqa: E402
from mdir_b200.qe import DBA_BLOCK  # noqa: E402
from mdir_b200.search import WIDE_Q  # noqa: E402

N, D, NQ, K, TRUNC, REPS, WARM = 1001001, 2048, 70, 50, 1000, 50, 5


def events(fn):
    out = []
    for _ in range(WARM):
        fn()
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        out.append((a, b))
    torch.cuda.synchronize()
    return np.array([a.elapsed_time(b) for a, b in out])


def main():
    dev = "cuda:0"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("# %s -- read in the same call" % card)
    print("# R1M shape: %d x %d unit randn rows, %d queries (db rows + noise), k = %d, trunc = %d" % (N, D, NQ, K, TRUNC))
    g = torch.Generator(device=dev).manual_seed(1234)
    db = torch.empty((N, D), dtype=torch.float32, device=dev)
    for r0 in range(0, N, 65536):
        blk = torch.randn((min(65536, N - r0), D), device=dev, generator=g)
        db[r0:r0 + blk.shape[0]] = blk / blk.norm(dim=1, keepdim=True)
    src = torch.randperm(N, device=dev, generator=g)[:NQ]
    q = db[src] + 0.5 * torch.randn((NQ, D), device=dev, generator=g) / D ** 0.5
    q = q / q.norm(dim=1, keepdim=True)
    index = mdir_b200.Index.from_packed(mdir_b200.search.pack_bf16(db), db32=db)
    index.search(q, 100, precision="fp32")
    torch.cuda.synchronize()

    t0 = time.perf_counter()
    dif = mdir_b200.Diffusion(index, k=K, gamma=3.0)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    nbr, S, deg = dif.graph()
    t0 = time.perf_counter()                       # the build's search passes alone, repeated
    for r0 in range(0, N, DBA_BLOCK):
        index.search(index.db32[r0:min(r0 + DBA_BLOCK, N)], K + 1, precision="fp32", block_q=WIDE_Q)
    torch.cuda.synchronize()
    t_knn = time.perf_counter() - t0
    n_edges = int((nbr >= 0).sum())
    print("build  %.3f s   (top-%d of %d rows + graph; %.1f mutual neighbours per row, %d isolated rows)"
          % (t_build, K + 1, N, n_edges / N, int((deg == 0).sum())))
    print("       %.3f s   of it: the top-%d search passes alone (timed again)" % (t_knn, K + 1))

    s, L = index.search(q, TRUNC, precision="fp32")
    t_search = events(lambda: index.search(q, TRUNC, precision="fp32"))
    lib = _lib.lib()
    ws_bytes = lib.mdir_diffusion_solve_workspace_bytes(NQ, TRUNC, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    f = torch.empty((NQ, 100), dtype=torch.float32, device=dev)
    ids = torch.empty((NQ, 100), dtype=torch.int32, device=dev)

    def solve():
        _lib.check(lib.mdir_diffusion_solve(_lib.ptr(L), _lib.ptr(s), NQ, TRUNC, _lib.ptr(index.slot_id), N, _lib.ptr(nbr), _lib.ptr(S), K,
                                            10, 3.0, 0.99, 20, 1e-6, 100, _lib.ptr(ws), ws_bytes, _lib.ptr(f), _lib.ptr(ids), _lib.stream()),
                   "mdir_diffusion_solve")
    t_solve = events(solve)
    steps = []
    for r in range(WARM + REPS):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fo, io = dif.search(q, k=100, trunc=TRUNC, k_q=10, alpha=0.99, iters=20, rtol=1e-6)
        torch.cuda.synchronize()
        if r >= WARM:
            steps.append((time.perf_counter() - t0) * 1e3)
    assert torch.equal(fo, f) and torch.equal(io, ids)
    print("search %.3f ms  (index.search(q, %d, fp32), median of %d; min %.3f)" % (np.median(t_search), TRUNC, REPS, t_search.min()))
    print("solve  %.3f ms  (mdir_diffusion_solve, %d queries, iters 20, median of %d; min %.3f)" % (np.median(t_solve), NQ, REPS, t_solve.min()))
    print("step   %.3f ms  (Diffusion.search end to end, host clock, median of %d)" % (np.median(steps), REPS))
    print("status words nonzero: %d of %d" % (int((dif.status() != 0).sum()), NQ))


if __name__ == "__main__":
    main()
