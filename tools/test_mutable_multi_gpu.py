#!/usr/bin/env python
"""Removal on a sharded index (run under torchrun on a box with >= 2 GPUs):

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29653 tools/test_mutable_multi_gpu.py

Every rank holds a row shard and makes the same ShardedIndex.remove / restore call with the same GLOBAL id list; the
sharded results must equal a single-GPU Index with the same removals bit for bit, in every exchange mode (NVLink
exchange sync / deferred / overlap, ncclAllGather route, CUDA graph, split graphs, SearchPipeline).  Rank 0 prints one
PASS/FAIL line per check and exits non-zero on failure."""
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
    n = 40000 * world                            # every shard large enough for the one-launch route (split graphs)
    db = synth.descriptors(n, 64, 581, clusters=200)
    q, src = synth.planted_queries(db, nq, 582)
    lo, hi = ShardedIndex.shard_bounds(n, world, rank)
    sharded = ShardedIndex(db[lo:hi], idx_base=lo, device=dev)
    single = mdir_b200.Index(db, device=dev)
    rs = np.random.RandomState(583)
    removed = np.sort(rs.choice(n, n // 3, replace=False))
    removed = np.unique(np.concatenate([removed, src]))          # the planted answers go too
    sharded.remove(removed)
    single.remove(removed)
    check("n_live of the shard", sharded.local.n_live == (hi - lo) - int(((removed >= lo) & (removed < hi)).sum()))
    for prec in ("bf16", "fp32"):
        ref = single.search(q, k, precision=prec)
        check("sync exchange after remove == single (%s)" % prec, same(sharded.search(q, k, precision=prec), ref))
    ref = single.search(q, k)
    check("removed ids never returned", not bool(np.isin(ref[1].cpu().numpy(), removed).any()))
    ShardedIndex.p2p = False
    nccl = ShardedIndex.from_local(sharded.local)
    ShardedIndex.p2p = True
    check("ncclAllGather route after remove == single", nccl._mb is None and same(nccl.search(q, k), ref))
    gs = GraphedSearch(sharded, nq, k)
    out = gs(torch.from_numpy(q).to(dev))
    torch.cuda.synchronize()
    check("CUDA graph after remove == single", same(out, ref) and not gs.check_overflow())
    gd = GraphedSearch(sharded, nq, k, deferred=True)
    gd(torch.from_numpy(q).to(dev))
    out = gd.drain()
    torch.cuda.synchronize()
    check("deferred-exchange graph after remove == single", same(out, ref))
    go = GraphedSearch(sharded, nq, k, overlap=True)
    out = go(torch.from_numpy(q).to(dev))
    torch.cuda.synchronize()
    check("overlap graph after remove == single", go.overlap and same(out, ref))
    gsp = GraphedSearch(sharded, nq, k, overlap=True, split=True)
    out = gsp(torch.from_numpy(q).to(dev))
    torch.cuda.synchronize()
    check("split graphs after remove == single (split=%s)" % gsp.split, gsp.split and same(out, ref))
    # restore half of the removed ids: the captured graphs see it without re-capture
    back = removed[::2]
    sharded.restore(back)
    single.restore(back)
    ref2 = single.search(q, k)
    good = True
    for g in (gs, go, gsp):
        out = g(torch.from_numpy(q).to(dev))
        torch.cuda.synchronize()
        good &= same(out, ref2)
    check("graphs after restore == single, no re-capture", good)
    # SearchPipeline: tickets before a remove see the old live set, tickets after it the new one
    hb = torch.from_numpy(q).pin_memory()
    more = removed[1::2][:500]
    tmp = mdir_b200.Index(db, device=dev)
    tmp.remove(np.setdiff1d(removed, back))
    tmp.remove(more)
    ref3 = tmp.search(q, k)
    for deferred in (False, True):
        pipe = mdir_b200.SearchPipeline(sharded, nq, k, deferred=deferred)
        t0 = pipe.submit(hb)
        pipe.remove(more)
        t1 = pipe.submit(hb)
        s0, i0 = pipe.result(t0)
        s0, i0 = s0.copy(), i0.copy()
        s1, i1 = pipe.result(t1)
        good = np.array_equal(i0, ref2[1].cpu().numpy()) and np.array_equal(s0, ref2[0].cpu().numpy())
        good &= np.array_equal(i1, ref3[1].cpu().numpy()) and np.array_equal(s1, ref3[0].cpu().numpy())
        check("SearchPipeline (%s exchange): ticket before remove == old, after == new" % ("deferred" if deferred else "overlap"), good)
        sharded.restore(more)
        del pipe
    try:
        sharded.remove([n + 5])
        raised = False
    except mdir_b200.MdirError:
        raised = True
    check("an id outside every shard raises on every rank", raised)
    check("exchange status clean", sharded.exchange_status() == 0)
    torch.cuda.synchronize()
    dist.barrier()
    sharded.close()
    if rank == 0:
        print("MUTABLE MULTI-GPU %s" % ("PASSED" if ok_all else "FAILED"), flush=True)
    sys.stdout.flush()
    os._exit(0 if ok_all else 1)


if __name__ == "__main__":
    main()
