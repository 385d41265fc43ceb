#!/usr/bin/env python
"""Compaction of a sharded index (run under torchrun on a box with >= 2 GPUs):

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29657 tools/test_compaction_multi_gpu.py

Every rank removes the same GLOBAL ids and calls ShardedIndex.compact() at the same point; each compacts its own shard,
ids unchanged.  The sharded results must equal a compacted single-GPU Index bit for bit in the sync and deferred
exchange modes and in the split / overlap serving graphs, also after a second removal and compaction.  Rank 0 prints
one PASS/FAIL line per check and exits non-zero on failure."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from oracle import synth  # noqa: E402
import mdir_b200  # noqa: E402
from mdir_b200.search import GraphedSearch, ShardedIndex  # noqa: E402


def main():
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dev = torch.device("cuda", lr)
    dist.init_process_group("nccl", device_id=dev)
    ok_all = True

    def check(name, cond):
        nonlocal ok_all
        flag = torch.tensor([1 if cond else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        good = bool(flag.item())
        ok_all &= good
        if rank == 0:
            print("[%s] %s" % ("PASS" if good else "FAIL", name), flush=True)

    def same(a, b):
        return torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])

    nq, k = 70, 100
    n = 40000 * world
    db = synth.descriptors(n, 64, 681, clusters=200)
    q, src = synth.planted_queries(db, nq, 682)
    lo, hi = ShardedIndex.shard_bounds(n, world, rank)
    sharded = ShardedIndex(db[lo:hi], idx_base=lo, device=dev)
    single = mdir_b200.Index(db, device=dev)
    graphs = {"split": GraphedSearch(sharded, nq, k, overlap=True, split=True)} if sharded._mb is not None else {}
    rs = np.random.RandomState(683)
    for rnd, frac in enumerate((0.3, 0.5)):
        live = single._ids[single._live_host[:single._n_used]]
        removed = np.sort(rs.choice(live, int(frac * live.size), replace=False))
        sharded.remove(removed)
        single.remove(removed)
        purged = sharded.compact()
        single.compact()
        check("round %d: shard purged its own removed rows" % rnd, purged == int(((removed >= lo) & (removed < hi)).sum()))
        check("round %d: shard extent == its live rows" % rnd, int(sharded.local.n_scan.item()) == sharded.local.n_live)
        for prec in ("bf16", "fp32"):
            ref = single.search(q, k, precision=prec)
            check("round %d: sync exchange == single compacted (%s)" % (rnd, prec), same(sharded.search(q, k, precision=prec), ref))
        ref = single.search(q, k)
        check("round %d: removed ids never returned" % rnd, not bool(np.isin(ref[1].cpu().numpy(), removed).any()))
        if sharded._mb is not None:
            sharded.search(q, k, exchange="deferred")
            got = sharded.drain(nq, k)
            check("round %d: deferred exchange == single compacted" % rnd, same(got, ref))
            gs = graphs["split"]
            out = gs(q)
            torch.cuda.synchronize()
            check("round %d: split graph captured before compaction == single compacted" % rnd, same(out, ref) and not gs.check_overflow())
        elif rank == 0 and rnd == 0:
            print("[SKIP] no peer-memory mailboxes: deferred and split modes not run", flush=True)
    sharded.close()
    dist.barrier()
    if rank == 0:
        print("COMPACTION MULTI-GPU PASSED" if ok_all else "COMPACTION MULTI-GPU FAILED", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if ok_all else 1)


if __name__ == "__main__":
    main()
