"""Offline diffusion (DiffusionTable) at the R1M shape of tools/time_diffusion.py (1,001,001 x 2048 unit randn rows,
70 queries, graph k = 50; table width = 100, trunc = 1000, alpha = 0.99, iters 20, rtol 1e-6; queries k = 100, k_q = 10;
one GPU).

  * build   -- Diffusion.offline(): host clock around the call plus a device synchronise, and its device time split into
               the search passes and the solves (DiffusionTable.timed, CUDA events), for each (OFFLINE_CHUNK,
               OFFLINE_BLOCK_Q) of SWEEP; every build's table is compared bit for bit with the first.
  * memory  -- the table's device bytes (8 width per slot of the capacity).
  * step    -- DiffusionTable.search(q) and Diffusion.search(q) end to end in the same process: host clock around the
               call plus a device synchronise, median over REPS.
  * parts   -- the k_q search index.search(q, 10, fp32) alone and mdir_diffusion_combine alone: CUDA events, median over REPS.

    python tools/time_diffusion_offline.py
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mdir_b200  # noqa: E402
import mdir_b200.diffusion as dmod  # noqa: E402
from mdir_b200 import _lib  # noqa: E402

N, D, NQ, K, WIDTH, TRUNC, KOUT, KQ, REPS, WARM = 1001001, 2048, 70, 50, 100, 1000, 100, 10, 50, 5
SWEEP = [(8192, 128), (32768, 128), (1024, 128), (8192, 256), (8192, 512), (8192, 1024)]      # (rows per chunk, queries per scan pass)


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


def host_ms(fn):
    out = []
    for r in range(WARM + REPS):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = fn()
        torch.cuda.synchronize()
        if r >= WARM:
            out.append((time.perf_counter() - t0) * 1e3)
    return np.array(out), res


def main():
    dev = "cuda:0"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("# %s -- read in the same call" % card)
    print("# R1M shape: %d x %d unit randn rows, %d queries (db rows + noise), graph k = %d; table width = %d, trunc = %d; "
          "queries k = %d, k_q = %d" % (N, D, NQ, K, WIDTH, TRUNC, KOUT, KQ))
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
    dif = mdir_b200.Diffusion(index, k=K, gamma=3.0)
    torch.cuda.synchronize()

    mdir_b200.DiffusionTable.timed = True
    tab = None
    for chunk, block_q in SWEEP:
        dmod.OFFLINE_CHUNK, dmod.OFFLINE_BLOCK_Q = chunk, block_q
        unc0 = index.cert["uncertified"]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        t = dif.offline(width=WIDTH, trunc=TRUNC, alpha=0.99, iters=20, rtol=1e-6)
        torch.cuda.synchronize()
        t_build = time.perf_counter() - t0
        bt = t.build_time
        if tab is None:
            tab, same = t, "first"
        else:
            same = torch.equal(t.tab_ids, tab.tab_ids) and torch.equal(t.tab_f.view(torch.int32), tab.tab_f.view(torch.int32))
            del t
        print("build  chunk %6d  block_q %4d  %7.2f s host   device: search passes %7.2f s, solves %6.3f s   "
              "uncertified rows %d   table bit-identical to the first: %s"
              % (chunk, block_q, t_build, bt["search"] / 1e3, bt["solve"] / 1e3, index.cert["uncertified"] - unc0, same))
    mdir_b200.DiffusionTable.timed = False
    nbytes = tab.tab_ids.numel() * 4 + tab.tab_f.numel() * 4
    print("table  %.1f MB on the device (%d slots x %d x 8 B)" % (nbytes / 1e6, tab.tab_ids.shape[0], WIDTH))

    t_off, (fo, io) = host_ms(lambda: tab.search(q, k=KOUT, k_q=KQ))
    st_off = int((tab.status() != 0).sum())
    t_on, (_, in_) = host_ms(lambda: dif.search(q, k=KOUT, trunc=TRUNC, k_q=KQ, alpha=0.99, iters=20, rtol=1e-6))
    s, L = index.search(q, KQ, precision="fp32")
    t_kq = events(lambda: index.search(q, KQ, precision="fp32"))
    lib = _lib.lib()
    f = torch.empty((NQ, KOUT), dtype=torch.float32, device=dev)
    ids = torch.empty((NQ, KOUT), dtype=torch.int32, device=dev)

    def combine():
        _lib.check(lib.mdir_diffusion_combine(_lib.ptr(L), _lib.ptr(s), NQ, KQ, _lib.ptr(index.slot_id), index._n_used, _lib.ptr(tab.tab_ids),
                                              _lib.ptr(tab.tab_f), WIDTH, 3.0, KOUT, _lib.ptr(f), _lib.ptr(ids), _lib.stream()),
                   "mdir_diffusion_combine")
    t_comb = events(combine)
    assert torch.equal(f.view(torch.int32), fo.view(torch.int32)) and torch.equal(ids, io)
    overlap = np.mean([np.intersect1d(a, b).size / KOUT for a, b in zip(io.cpu().numpy(), in_.cpu().numpy())])
    print("step   %.3f ms  (DiffusionTable.search end to end, host clock + sync, median of %d; min %.3f)" % (np.median(t_off), REPS, t_off.min()))
    print("       %.3f ms  (Diffusion.search end to end, trunc %d, same process, median of %d; min %.3f)"
          % (np.median(t_on), TRUNC, REPS, t_on.min()))
    print("parts  %.3f ms  (index.search(q, %d, fp32) alone, CUDA events, median of %d; min %.3f)" % (np.median(t_kq), KQ, REPS, t_kq.min()))
    print("       %.3f ms  (mdir_diffusion_combine alone, %d queries, CUDA events, median of %d; min %.3f)"
          % (np.median(t_comb), NQ, REPS, t_comb.min()))
    print("status words nonzero: %d of %d (k_q search); top-%d overlap with Diffusion.search %.3f" % (st_off, NQ, KOUT, overlap))


if __name__ == "__main__":
    main()
