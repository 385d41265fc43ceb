"""Search step time of a mutable index before and after Index.compact() at the R1M shape (1,001,001 x 2048 unit randn
rows, 70 unit queries, top-100, certified fp32, one GPU), for both first passes: int8 (the default at this size) and
bf16 (int8 route disabled through search.I8_MIN_ROWS).

Per removed fraction (0, 10, 50, 90 %), before and after compact():
  * eager  -- index.search(check=True) per step, CUDA events over REPS steps after warm-up;
  * graph  -- replay of the split serving graphs (GraphedSearch(split=True): scan | finalize + re-score) captured BEFORE
              the compaction and replayed after it without re-capture;
  * scan   -- the first-pass scan kernel alone (CUDA events around its launch) and its rate on the bytes it scans:
              n_scan rows x (D B int8 + 4 B scale, or 2 D B bf16);
  * recovery -- status words of one check=False step (overflowed / uncertified queries) and whether a check=True step
              redid a block (int8 -> bf16, widening, dense);
and compact()'s wall time (host clock around the call and a device synchronise) with its effective bandwidth: the
bytes its schedule reads and writes (direct chunks once, staged chunks twice) plus the zeroed tail.

    python tools/time_compaction.py
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mdir_b200 import search  # noqa: E402

N, D, NQ, K, REPS = 1001001, 2048, 70, 100, 200


def _db(n, dev):
    g = torch.Generator(device=dev).manual_seed(1234)
    db = torch.empty((n, D), dtype=torch.float32, device=dev)
    for r0 in range(0, n, 65536):
        blk = torch.randn((min(65536, n - r0), D), device=dev, generator=g)
        db[r0:r0 + blk.shape[0]] = blk / blk.norm(dim=1, keepdim=True)
    return db


class ScanTimer:
    """Index.prof hook: CUDA events around the first-pass scan launch of every search."""

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
        return float(np.median(t))


def _events(fn, reps):
    for _ in range(10):
        fn()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for r in range(reps):
        fn(r)
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps


def _measure(index, gs, q):
    index.search(q[0], K, check=False)
    torch.cuda.synchronize()
    st = index.status().cpu().numpy()
    flagged = (int((st & 1).astype(bool).sum()), int((st & 2).astype(bool).sum()))
    c0 = dict(index.cert)
    eager = _events(lambda r=0: index.search(q[r % 8], K), REPS)
    redone = (index.cert["int8_redone"] - c0["int8_redone"]) + (index.cert["widened_blocks"] - c0["widened_blocks"])
    graph = _events(lambda r=0: gs(q[r % 8]), REPS)
    gs_ok = not gs.check_overflow()
    timer = ScanTimer()
    index.prof = timer
    for r in range(50):
        index.search(q[r % 8], K, check=False)
    index.prof = None
    scan = timer.ms()
    n_scan = int(index.n_scan.item())
    scan_bytes = n_scan * (D + 4) if index.route == "int8" else n_scan * 2 * D
    return eager, graph, scan, scan_bytes / (scan * 1e-3) / 1e12, flagged, redone, gs_ok


def _schedule_bytes(index):
    used = index._live_host[:index._n_used]
    rb = 2 * D + (4 * D if index.db32 is not None else 0) + (D + 4 if index.db8 is not None else 0) + 4
    moved = sum((4 if st else 2) * n_dst for _, _, _, n_dst, st in search.compaction_schedule(used, index.compact_chunk))
    return (moved + (index._n_used - int(used.sum()))) * rb


def main():
    dev = torch.device("cuda", 0)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          stdout=subprocess.PIPE).stdout.decode().strip()
    print("# %s -- read in the same run" % card, flush=True)
    gq = torch.Generator(device="cpu").manual_seed(99)
    q = torch.randn((8, NQ, D), generator=gq)
    q = (q / q.norm(dim=2, keepdim=True)).to(dev)
    db = _db(N, dev)
    i8_min = search.I8_MIN_ROWS
    for first in ("int8", "bf16"):
        search.I8_MIN_ROWS = i8_min if first == "int8" else 1 << 40
        for frac in (0.0, 0.1, 0.5, 0.9):
            index = search.Index(db.clone(), device=dev)        # the index's master copy: compact() rewrites it
            if frac:
                index.remove(np.random.RandomState(7).choice(N, int(frac * N), replace=False))
            gs = search.GraphedSearch(index, NQ, K, overlap=True, split=True)
            for phase in ("before", "after"):
                if phase == "after":
                    nbytes = _schedule_bytes(index)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    purged = index.compact()
                    torch.cuda.synchronize()
                    dt = time.perf_counter() - t0
                    if purged:
                        print("  compact(): %d rows purged in %.1f ms, %.2f TB/s effective (%.1f GB read + written)" %
                              (purged, dt * 1e3, nbytes / dt / 1e12, nbytes / 1e9), flush=True)
                    else:
                        print("  compact(): nothing removed, %.3f ms (no launch)" % (dt * 1e3), flush=True)
                eager, graph, scan, tbs, (ovf, unc), redone, gs_ok = _measure(index, gs, q)
                print("first pass %-4s %3d%% removed %-6s  n_scan %8d  eager %.3f ms  split graph %.3f ms  scan %.3f ms "
                      "(%.2f TB/s on scanned bytes)  route %s  check=False step: %d/%d overflowed, %d/%d uncertified  "
                      "recovery blocks %d  graph status clear %s" %
                      (first, int(frac * 100), phase, int(index.n_scan.item()), eager, graph, scan, tbs, index.route, ovf, NQ,
                       unc, NQ, redone, gs_ok), flush=True)
            del gs, index
            torch.cuda.empty_cache()
    search.I8_MIN_ROWS = i8_min


if __name__ == "__main__":
    main()
