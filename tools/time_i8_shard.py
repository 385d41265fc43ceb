"""Int8 vs bf16 first pass of the certified fp32 search by shard size (the per-rank shards of the 1/2/4/8-GPU bench).

For each shard size: the bench's data (unit randn rows at D = 2048, 8 batches of 70 unit queries, top-100), the
local step (pack, fused scan, finalize + certified re-score) through each route, check=False as in the serving
graphs.  Prints per size: queries whose certificate failed on each route, and the step time of each (CUDA events,
mean over 8 x REPS steps).  The int8 route's minimum shard size (search.I8_MIN_ROWS) is lifted for the run.

    python tools/time_i8_shard.py [rows ...]
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mdir_b200 import search  # noqa: E402

D, NQ, K, REPS = 2048, 70, 100, 20


def main():
    sizes = [int(a) for a in sys.argv[1:]] or [125126, 250252, 500501, 1001001]
    search.I8_MIN_ROWS = 0
    dev = torch.device("cuda", 0)
    gq = torch.Generator(device="cpu").manual_seed(99)
    q = torch.randn((8, NQ, D), generator=gq)
    q = (q / q.norm(dim=2, keepdim=True)).to(dev)
    print(torch.cuda.get_device_name(0))
    for n in sizes:
        g = torch.Generator(device=dev).manual_seed(1234)
        db = torch.empty((n, D), dtype=torch.float32, device=dev)
        for r0 in range(0, n, 65536):
            blk = torch.randn((min(65536, n - r0), D), device=dev, generator=g)
            db[r0:r0 + blk.shape[0]] = blk / blk.norm(dim=1, keepdim=True)
        index = search.Index.from_packed(search.pack_bf16(db), db32=db)
        index.stats()
        db8 = index.db8
        res = {}
        for route in ("int8", "bf16"):
            index.db8 = db8 if route == "int8" else None
            failed = 0
            for b in range(8):
                index.search(q[b], K, precision="fp32", check=False)
                failed += int(index.status().ne(0).sum().item())
            assert index.route == route
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            torch.cuda.synchronize()
            ev[0].record()
            for r in range(REPS * 8):
                index.search(q[r % 8], K, precision="fp32", check=False)
            ev[1].record()
            torch.cuda.synchronize()
            res[route] = (failed, ev[0].elapsed_time(ev[1]) / (REPS * 8))
        print("rows %8d  int8: %3d/%d uncertified, %.3f ms/step   bf16: %3d/%d uncertified, %.3f ms/step" %
              (n, res["int8"][0], 8 * NQ, res["int8"][1], res["bf16"][0], 8 * NQ, res["bf16"][1]), flush=True)
        del index, db, db8
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
