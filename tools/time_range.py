"""Index.range_search at the R1M shape (1,001,001 x 2048 unit randn rows, 70 queries, one GPU), next to search(k=100).

Per-query thresholds are set from the fp32 scores of every row (Index.scores(precision="fp32") and mdir's own top-k) so
that each query has about 100, 1,000 and 10,000 matches.  For each target and both precisions:
  * step   -- range_search(q, min_score) per 70-query step: host clock around the call, which ends in its own read-back
              of the survivor counts plus a final device synchronise; median and mean over REPS steps after warm-up;
  * scan   -- the FILTER scan kernel alone (CUDA events around its launch, through the Index.prof hook) and its rate on
              the bytes it scans (n_used rows x 2 D B of bf16);
  * rescans -- steps that needed the exact re-scan (a candidate segment overflowed), out of warm-up + REPS;
  * rows   -- matches per query (mean) and candidates per query that the scan passed, survivors/candidates.
The search(k=100, precision="fp32") line is the eager certified top-k step of the same index and queries.  Last, one
min_score = -inf call over NQ_ALL queries at both precisions (every row returned: the exact re-scan, then the group
sort + merge of a query with more than 16,384 survivors), next to Index.ranks over the same queries.

    python tools/time_range.py
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mdir_b200  # noqa: E402

N, D, NQ, REPS, WARM = 1001001, 2048, 70, 50, 5
NQ_ALL = 8          # queries of the min_score = -inf call (8 M results of 8 B + the fp32 gather of 8 x 8 GB)
TARGETS = (100, 1000, 10000)


class ScanTimer:
    """Index.prof hook: CUDA events around every scan launch."""

    def __init__(self):
        self.pairs = []

    def begin(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.pairs.append([e, None])

    def end(self, _bytes):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.pairs[-1][1] = e

    def ms(self):
        torch.cuda.synchronize()
        t = [a.elapsed_time(b) for a, b in self.pairs]
        self.pairs = []
        return t


def main():
    dev = "cuda:0"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("# %s -- read in the same call" % card)
    print("# R1M shape: %d x %d unit randn rows, %d queries (db rows + noise), REPS %d after %d warm-up steps" % (N, D, NQ, REPS, WARM))
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
    _, val = mdir_b200.topk_from_scores(dense.t().contiguous(), max(TARGETS))
    val = val.cpu().numpy()                                   # (k, nq), descending
    del dense
    index._db_x3 = None
    torch.cuda.empty_cache()
    scan_bytes = index._n_used * D * 2

    def run(fn):
        for _ in range(WARM):
            fn()
        torch.cuda.synchronize()
        t = []
        for _ in range(REPS):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            t.append((time.perf_counter() - t0) * 1e3)
        return np.array(t)

    t = run(lambda: index.search(q, 100, precision="fp32"))
    print("search(k=100, fp32)          step median %.3f ms  mean %.3f ms  route %s" % (np.median(t), t.mean(), index.route))
    for precision in ("fp32", "bf16"):
        for target in TARGETS:
            thr = torch.from_numpy(val[target - 1].copy())
            r0 = dict(index.range_stats)
            t = run(lambda: index.range_search(q, thr, precision=precision))
            rescans = index.range_stats["rescans"] - r0["rescans"]
            # one instrumented step: the scan kernel alone, the candidate count and the result size
            prof = ScanTimer()
            index.prof = prof
            lims, _, _ = index.range_search(q, thr, precision=precision)
            scan_ms = prof.ms()
            index.prof = None
            cand = int(index._buf("range_segcnt", (128, 149), torch.int32)[:NQ].sum())
            rows = int(lims[-1])
            print("range %s ~%5d / query    step median %.3f ms  mean %.3f ms  | scan %.3f ms  %.2f TB/s  | re-scanned steps %d of %d"
                  "  | matches %.0f / query, scan candidates %.0f / query (%.2f kept), large sorts %d"
                  % (precision, target, np.median(t), t.mean(), scan_ms[0], scan_bytes / scan_ms[0] / 1e9, rescans, WARM + REPS,
                     rows / NQ, cand / NQ, rows / max(1, cand), index.range_stats["large_sorts"] - r0["large_sorts"]))
    # min_score = -inf: every row of every query comes back (1,001,001 per query), through the exact re-scan and the
    # group sort + merge of queries with more than 16,384 survivors; next to Index.ranks, the full ranking, for scale
    qn = q[:NQ_ALL]
    for precision in ("bf16", "fp32"):
        index.range_search(qn, float("-inf"), precision=precision)
        r0 = dict(index.range_stats)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        lims, _, _ = index.range_search(qn, float("-inf"), precision=precision)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        print("range %s min_score=-inf, %d queries: %.1f ms (%.2f ms per query), %d rows per query, re-scan groups %d, large sorts %d"
              % (precision, NQ_ALL, dt, dt / NQ_ALL, int(lims[1] - lims[0]), index.range_stats["rescan_groups"] - r0["rescan_groups"],
                 index.range_stats["large_sorts"] - r0["large_sorts"]))
        del lims
    index.ranks(qn)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    index.ranks(qn)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) * 1e3
    print("Index.ranks (bf16 full ranking), %d queries: %.1f ms (%.2f ms per query)" % (NQ_ALL, dt, dt / NQ_ALL))
    print("range_stats %s" % index.range_stats)


if __name__ == "__main__":
    main()
