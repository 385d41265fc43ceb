"""Search step time of a mutable index at the R1M shape (1,001,001 x 2048 unit randn rows, 70 unit queries, top-100,
one GPU), for both first passes of the certified fp32 search: int8 (the default at this size) and bf16 (int8 route
disabled through search.I8_MIN_ROWS).

Cases: 0 %, 1 %, 10 % and 50 % of the rows removed, and a 5 % free-capacity tail (Index(db, capacity=1.05 n)).  Per
case: the step time of index.search(check=True) -- the serving answer including any recovery -- as CUDA events over
REPS steps after warm-up, and the status words of one check=False step (how many queries the first pass flagged: bit 0
= a candidate segment overflowed, bit 1 = certificate failed), which is what a captured graph would hand to the
pipeline's recovery.  Then the host-to-result time of add() of 10 k rows and remove() of 10 k ids (synchronised).

    python tools/time_mutable.py
"""
import os
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


def _step(index, q):
    index.search(q[0], K, precision="fp32", check=False)
    torch.cuda.synchronize()
    st = index.status().cpu().numpy()
    flagged = (int((st & 1).astype(bool).sum()), int((st & 2).astype(bool).sum()))
    for r in range(10):
        index.search(q[r % 8], K, precision="fp32")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for r in range(REPS):
        index.search(q[r % 8], K, precision="fp32")
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / REPS, flagged, index.route


def main():
    dev = torch.device("cuda", 0)
    print("# %s" % torch.cuda.get_device_name(0), flush=True)
    gq = torch.Generator(device="cpu").manual_seed(99)
    q = torch.randn((8, NQ, D), generator=gq)
    q = (q / q.norm(dim=2, keepdim=True)).to(dev)
    db = _db(N, dev)
    i8_min = search.I8_MIN_ROWS
    for first in ("int8", "bf16"):
        search.I8_MIN_ROWS = i8_min if first == "int8" else 1 << 40
        for case in ("0%", "1%", "10%", "50%", "tail5%"):
            if case == "tail5%":
                index = search.Index(db, device=dev, capacity=int(N * 1.05))
            else:
                index = search.Index(db, device=dev)
                frac = float(case[:-1]) / 100
                if frac:
                    index.remove(np.random.RandomState(7).choice(N, int(frac * N), replace=False))
            ms, (ovf, unc), route = _step(index, q)
            print("first pass %-4s  %-7s live %8d of %8d slots  %.3f ms/step  route %-4s  check=False step: %2d/%d overflowed, "
                  "%2d/%d uncertified" % (first, case, index.n_live, index.n, ms, route, ovf, NQ, unc, NQ), flush=True)
            del index
            torch.cuda.empty_cache()
    search.I8_MIN_ROWS = i8_min
    index = search.Index(db[:N - 10000], device=dev, capacity=N)
    index.search(q[0], K)                                   # stats and int8 plane exist: add() merges into them
    new = db[N - 10000:].clone()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ids = index.add(new)
    torch.cuda.synchronize()
    t_add = time.perf_counter() - t0
    rm = np.random.RandomState(8).choice(N, 10000, replace=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    index.remove(rm)
    torch.cuda.synchronize()
    t_rm = time.perf_counter() - t0
    print("add() of 10,000 rows (device fp32 in): %.2f ms;  remove() of 10,000 host ids: %.2f ms  (ids %d..%d)" %
          (t_add * 1e3, t_rm * 1e3, int(ids[0]), int(ids[-1])), flush=True)


if __name__ == "__main__":
    main()
