"""Incremental diffusion-graph updates at the R1M shape (1,001,001 x 2048 unit randn rows, capacity + 10,000, k = 50, one
GPU), against the build.

  * build                 -- Diffusion(index, k=50): host clock around the constructor plus a device synchronise (the
                             index's one-time certificate pass runs in a search before it, so it is not counted).
  * add / remove / restore / compact through the Diffusion: host clock around the call plus a device synchronise, and
                             the device time of each phase (CUDA events, Diffusion.timed): search = the build's search
                             of the rows whose lists are redone, scan = mdir_sim_scan_dense_bf16 of the batch against
                             the rows, merge = mdir_diffusion_merge, stale = mdir_diffusion_stale_rows, graph =
                             mdir_diffusion_graph + _normalize.  Counters: Diffusion.update_stats, per call.
  * Sequence: add 1, add 1,024; remove 10 / 100 / 1,000 / 10,000 random live rows, each followed by the restore of the
    same rows; remove 10,000, compact, add 10,000 into the freed slots.  Then a new Diffusion over the final index and a
    bitwise comparison of the raw lists, graph() and search() against it.

    python tools/time_diffusion_update.py
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mdir_b200  # noqa: E402

N, D, K, EXTRA, NQ = 1001001, 2048, 50, 10000, 70


def unit_randn(n, gen, dev):
    out = torch.empty((n, D), dtype=torch.float32, device=dev)
    for r0 in range(0, n, 65536):
        blk = torch.randn((min(65536, n - r0), D), device=dev, generator=gen)
        out[r0:r0 + blk.shape[0]] = blk / blk.norm(dim=1, keepdim=True)
    return out


def main():
    dev = "cuda:0"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("# %s -- read in the same call" % card)
    print("# R1M shape: %d x %d unit randn rows, capacity + %d, k = %d" % (N, D, EXTRA, K))
    gen = torch.Generator(device=dev).manual_seed(1234)
    db = unit_randn(N, gen, dev)
    new = unit_randn(1 + 1024 + 10000, gen, dev)
    src = torch.randperm(N, device=dev, generator=gen)[:NQ]
    q = db[src] + 0.5 * torch.randn((NQ, D), device=dev, generator=gen) / D ** 0.5
    q = q / q.norm(dim=1, keepdim=True)
    index = mdir_b200.Index(db, device=dev, capacity=N + EXTRA)
    del db
    index.search(q, 100, precision="fp32")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    g = mdir_b200.Diffusion(index, k=K, gamma=3.0)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    print("build                 %10.1f ms" % (t_build * 1e3))
    g.timed = True
    rs = np.random.RandomState(5)

    def op(name, fn):
        before = dict(g.update_stats)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        ph = "  ".join("%s %.1f" % (k, v) for k, v in sorted(g.update_time.items()))
        st = "  ".join("%s %d" % (k, g.update_stats[k] - before[k]) for k in g.update_stats)
        print("%-21s %10.1f ms  (x%.0f faster than the build)  device ms: %s  | %s" % (name, dt * 1e3, t_build / dt, ph, st))
        return r

    op("add 1", lambda: g.add(new[:1]))
    op("add 1024", lambda: g.add(new[1:1025]))
    for n_rm in (10, 100, 1000, 10000):
        live = index._ids[index._live_host[:index._n_used]]
        ids = rs.choice(live, n_rm, replace=False)
        op("remove %d" % n_rm, lambda: g.remove(ids))
        op("restore %d" % n_rm, lambda: g.restore(ids))
    ids = rs.choice(index._ids, 10000, replace=False)
    op("remove 10000", lambda: g.remove(ids))
    op("compact", g.compact)
    op("add 10000 (freed)", lambda: g.add(new[1025:]))

    t0 = time.perf_counter()
    fresh = mdir_b200.Diffusion(index, k=K, gamma=3.0)
    torch.cuda.synchronize()
    print("fresh build           %10.1f ms" % ((time.perf_counter() - t0) * 1e3))
    n = index._n_used
    same_lists = torch.equal(g.knn_i[:n], fresh.knn_i[:n]) and torch.equal(g.knn_s[:n].view(torch.int32), fresh.knn_s[:n].view(torch.int32))
    same_graph = all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(g.graph(), fresh.graph()))
    f1, i1 = g.search(q)
    s1 = g.status().clone()
    f2, i2 = fresh.search(q)
    same_search = torch.equal(f1.view(torch.int32), f2.view(torch.int32)) and torch.equal(i1, i2) and torch.equal(s1, fresh.status())
    print("bitwise against the fresh build: lists %s, graph %s, search (f, ids, status) %s" % (same_lists, same_graph, same_search))
    if not (same_lists and same_graph and same_search):
        sys.exit(1)


if __name__ == "__main__":
    main()
