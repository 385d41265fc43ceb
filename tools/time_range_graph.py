"""Captured range serving at the R1M shape (1,001,001 x 2048 unit randn rows, 70 queries, one GPU): eager
Index.range_search next to GraphedRangeSearch and RangePipeline.

Per-query thresholds come from the fp32 scores of every row (as in tools/time_range.py), so that each query has about
100, 1,000 and 10,000 matches; max_results is 1,024 / 2,048 / 16,384 for the three targets.  For each target and both
precisions:
  * eager    -- range_search(q, min_score) per 70-query step: host clock around the call plus a device synchronise
                (the call itself reads the survivor counts back once); median over REPS steps after warm-up;
  * replay   -- GraphedRangeSearch: CUDA events around REPLAYS back-to-back replays of one graph (device time per step,
                no copies); flagged = queries the graph left to recovery in one replay;
  * pipeline -- RangePipeline at depth 2 and 3: TICKETS tickets from pinned host buffers (queries + thresholds up, the
                full lims / status / max_results arenas down), host clock from the first submit to the last result();
                steps/s, and how many tickets needed an eager recovery.
The D2H of one ticket is 70 * max_results * 8 B of arenas (+ lims and status).

    python tools/time_range_graph.py
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mdir_b200  # noqa: E402

N, D, NQ, REPS, WARM, REPLAYS, TICKETS = 1001001, 2048, 70, 50, 5, 200, 200
TARGETS = ((100, 1024), (1000, 2048), (10000, 16384))     # (matches per query, max_results)


def main():
    dev = "cuda:0"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("# %s -- read in the same call" % card)
    print("# R1M shape: %d x %d unit randn rows, %d queries (db rows + noise); eager %d steps after %d warm-up, %d replays, %d tickets"
          % (N, D, NQ, REPS, WARM, REPLAYS, TICKETS))
    g = torch.Generator(device=dev).manual_seed(1234)
    db = torch.empty((N, D), dtype=torch.float32, device=dev)
    for r0 in range(0, N, 65536):
        blk = torch.randn((min(65536, N - r0), D), device=dev, generator=g)
        db[r0:r0 + blk.shape[0]] = blk / blk.norm(dim=1, keepdim=True)
    src = torch.randperm(N, device=dev, generator=g)[:NQ]
    q = db[src] + 0.5 * torch.randn((NQ, D), device=dev, generator=g) / D ** 0.5
    q = q / q.norm(dim=1, keepdim=True)
    index = mdir_b200.Index.from_packed(mdir_b200.search.pack_bf16(db), db32=db)
    dense = index.scores(q, precision="fp32")
    _, val = mdir_b200.topk_from_scores(dense.t().contiguous(), max(t for t, _ in TARGETS))
    val = val.cpu().numpy()                                   # (k, nq), descending
    del dense
    index._db_x3 = None
    torch.cuda.empty_cache()
    qh = q.cpu().pin_memory()

    for precision in ("fp32", "bf16"):
        for target, max_results in TARGETS:
            thr = val[target - 1].copy()
            thr_t = torch.from_numpy(thr)
            for _ in range(WARM):
                index.range_search(q, thr_t, precision=precision)
            torch.cuda.synchronize()
            t = []
            for _ in range(REPS):
                t0 = time.perf_counter()
                lims, _, _ = index.range_search(q, thr_t, precision=precision)
                torch.cuda.synchronize()
                t.append((time.perf_counter() - t0) * 1e3)
            eager = float(np.median(t))
            rows = int(lims[-1])

            gr = mdir_b200.GraphedRangeSearch(index, NQ, max_results=max_results, precision=precision)
            gr(q, thr)
            torch.cuda.synchronize()
            flagged = int((gr.status != 0).sum())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(REPLAYS):
                gr.graph.replay()
            e1.record()
            torch.cuda.synchronize()
            replay = e0.elapsed_time(e1) / REPLAYS
            del gr

            pipe_txt = []
            for depth in (2, 3):
                pipe = mdir_b200.RangePipeline(index, NQ, max_results=max_results, depth=depth, precision=precision)
                for _ in pipe.map([(qh, thr)] * (2 * depth)):
                    pass
                n0 = pipe.n_recovered
                t0 = time.perf_counter()
                for _ in pipe.map([(qh, thr)] * TICKETS):
                    pass
                dt = time.perf_counter() - t0
                pipe_txt.append("depth %d %.0f steps/s (%.3f ms/step), recovered %d of %d"
                                % (depth, TICKETS / dt, dt / TICKETS * 1e3, pipe.n_recovered - n0, TICKETS))
                del pipe
            torch.cuda.empty_cache()
            print("range %s ~%5d / query (max_results %5d, %.0f matches / query)  eager %.3f ms  | replay %.3f ms, %d queries flagged"
                  "  | pipeline %s  | D2H %.2f MB / ticket"
                  % (precision, target, max_results, rows / NQ, eager, replay, flagged, "; ".join(pipe_txt),
                     NQ * max_results * 8 / 1e6))


if __name__ == "__main__":
    main()
