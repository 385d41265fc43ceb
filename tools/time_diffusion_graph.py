"""Captured diffusion serving (GraphedDiffusion, DiffusionPipeline) at the R1M shape of tools/time_diffusion.py
(1,001,001 x 2048 unit randn rows, graph k = 50, 70 queries; online trunc 1,000, k_q 10; table width 100, trunc 1,000,
k_q 10; k = 100, alpha 0.99, iters 20, rtol 1e-6; one GPU), for both sources:

  * eager    -- source.search(q) end to end: host clock around the call plus a device synchronise, median over REPS.
  * replay   -- GraphedDiffusion: CUDA events around REPLAYS back-to-back replays of one graph, per step; median of WINDOWS.
  * pipeline -- DiffusionPipeline.map over TICKETS tickets from pinned host buffers (upload, replay, download and the
                recovery of flagged queries), host clock from the first submit to the last result, per ticket; depth 2, 3.

Every replayed and pipelined result is compared bit for bit with the eager call on the same batch (a query the graph
flags is compared after the pipeline's recovery; the replay gives it no rows).  At this shape the shortlist search
takes the int8 first pass, which the test suite's small databases do not reach.

    python tools/time_diffusion_graph.py
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mdir_b200  # noqa: E402

N, D, NQ, K, WIDTH, TRUNC, KOUT, KQ = 1001001, 2048, 70, 50, 100, 1000, 100, 10
PARAMS = dict(alpha=0.99, iters=20, rtol=1e-6)
REPS, WARM, REPLAYS, WINDOWS, TICKETS, BATCHES = 50, 5, 200, 5, 240, 4


def host_ms(fn):
    out = []
    for r in range(WARM + REPS):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        if r >= WARM:
            out.append((time.perf_counter() - t0) * 1e3)
    return np.array(out)


def same(a, b):
    return np.array_equal(np.asarray(a[0]).view(np.int32), np.asarray(b[0]).view(np.int32)) and np.array_equal(a[1], b[1])


def run(name, src, p, batches, index):
    ref = [tuple(t.cpu().numpy() for t in src.search(b, k=KOUT, **p)) for b in batches]
    t_eager = host_ms(lambda: src.search(batches[0], k=KOUT, **p))
    gd = mdir_b200.GraphedDiffusion(src, NQ, KOUT, **p)
    flagged = 0
    for b, r in zip(batches, ref):
        f, ids = gd(b)
        f, ids, st = f.cpu().numpy(), ids.cpu().numpy(), gd.status.cpu().numpy()
        ok = st == 0
        flagged += int((~ok).sum())
        assert same((f[ok], ids[ok]), (r[0][ok], r[1][ok])), "%s: replay differs from eager" % name
        assert (ids[~ok] == -1).all() and np.isneginf(f[~ok]).all()
    for _ in range(WARM):
        gd()
    win = []
    for _ in range(WINDOWS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(REPLAYS):
            gd.graph.replay()
        b.record()
        b.synchronize()
        win.append(a.elapsed_time(b) / REPLAYS)
    win = np.array(win)
    print("%-7s eager    %.3f ms  (source.search end to end, host clock + sync, median of %d; min %.3f)"
          % (name, np.median(t_eager), REPS, t_eager.min()))
    print("%-7s replay   %.3f ms  (CUDA events, %d back-to-back replays per window, median of %d windows; min %.3f)   "
          "bit-identical to eager on %d batches: True   flagged queries in the replays %d"
          % (name, np.median(win), REPLAYS, WINDOWS, win.min(), len(batches), flagged))
    del gd
    for depth in (2, 3):
        pipe = mdir_b200.DiffusionPipeline(src, NQ, KOUT, depth=depth, **p)
        for i, out in enumerate(pipe.map(batches * 2)):                   # warm-up, and the results checked
            assert same(out, ref[i % len(batches)]), "%s: pipeline differs from eager" % name
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = 0
        for _ in pipe.map(batches[i % len(batches)] for i in range(TICKETS)):
            n += 1
        dt = (time.perf_counter() - t0) * 1e3 / n
        print("%-7s pipeline depth %d  %.3f ms per ticket  (host clock over %d tickets from pinned buffers; tickets redone %d)"
              % (name, depth, dt, n, pipe.n_recovered))
        del pipe


def main():
    dev = "cuda:0"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("# %s -- name, power limit, max SM clock, read in the same call" % card)
    print("# R1M shape: %d x %d unit randn rows, %d queries (db rows + noise), graph k = %d; online trunc %d, k_q %d; "
          "table width %d, trunc %d, k_q %d; k = %d" % (N, D, NQ, K, TRUNC, KQ, WIDTH, TRUNC, KQ, KOUT))
    g = torch.Generator(device=dev).manual_seed(1234)
    db = torch.empty((N, D), dtype=torch.float32, device=dev)
    for r0 in range(0, N, 65536):
        blk = torch.randn((min(65536, N - r0), D), device=dev, generator=g)
        db[r0:r0 + blk.shape[0]] = blk / blk.norm(dim=1, keepdim=True)
    batches = []
    for _ in range(BATCHES):
        src = torch.randperm(N, device=dev, generator=g)[:NQ]
        q = db[src] + 0.5 * torch.randn((NQ, D), device=dev, generator=g) / D ** 0.5
        batches.append((q / q.norm(dim=1, keepdim=True)).cpu().pin_memory())
    index = mdir_b200.Index.from_packed(mdir_b200.search.pack_bf16(db), db32=db)
    index.search(batches[0], 100, precision="fp32")
    print("# shortlist route: %s" % index.route)
    t0 = time.perf_counter()
    dif = mdir_b200.Diffusion(index, k=K, gamma=3.0)
    tab = dif.offline(width=WIDTH, trunc=TRUNC, **PARAMS)
    torch.cuda.synchronize()
    print("# graph + table built in %.1f s" % (time.perf_counter() - t0))
    run("online", dif, dict(trunc=TRUNC, k_q=KQ, **PARAMS), batches, index)
    run("table", tab, dict(k_q=KQ), batches, index)


if __name__ == "__main__":
    main()
