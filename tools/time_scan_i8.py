"""The fused first-pass scans alone at the bench shape: the int8 scan (sim_scan_kernel<kKindI8>) against the bf16 scan
(sim_scan_kernel<kKindBf16>), both in FUSED mode (threshold exchange + filter in one launch).

bench.py's data (1,001,001 unit randn rows at D = 2048, 70 unit queries of batch 0, top-100 with its shortlist depth),
Index.from_packed with the fp32 master, so the int8 plane exists; the int8 operand comes from Index._pack_q_i8 and
the bf16 one from pack_bf16.  Each launch is timed by CUDA events over REPS back-to-back launches, 3 rounds, the two
kinds alternating.  Printed per launch:
  - ms;
  - HBM bytes per second: the bytes the scan must stream (int8 rows + their fp32 scales, or bf16 rows) over the time;
  - shared-memory ingest bytes per SM per second: the bytes TMA writes into shared memory over (CTAs x time), from
    the shapes: for each CTA, (bytes staged per k-block of an MMA item) x k-blocks x items, summed over the grid.
    bf16 stages a 256-row tile (32 KB) plus the query block (n_pad x 128 B) per k-block of a tile.  int8 stages the
    database rows of the item plus both query planes (2 x n_pad x 128 B) per k-block; --i8-halves gives how many
    128-row halves the int8 kernel stages per item: 2 (the kernel as it is: one 256-row tile per item) or 3 (a kernel
    that groups a CTA's halves by three after the sample tile, as measured in profiles/r11_scan_i8_1gpu.log).
The card's name, power limit and SM clocks are read in the same run.

    python tools/time_scan_i8.py [--i8-halves 2]
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from mdir_b200.search import Index, pack_bf16, default_shortlist  # noqa: E402

REPS = 200
ROUNDS = 3
TILE = 256
NUM_SMS = 148


def smi():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip()


def balanced_grid(n_work, max_ctas):
    """common.cuh:balanced_grid."""
    if n_work <= max_ctas:
        return n_work
    rounds = -(-n_work // max_ctas)
    return -(-n_work // rounds)


def fused_ingest(n, D, nq, i8, i8_halves):
    """-> (CTAs, shared-memory bytes TMA writes over the whole launch) of one FUSED launch over n rows."""
    n_tiles = -(-n // TILE)
    g = balanced_grid(n_tiles, min(NUM_SMS, n_tiles // 2))
    n_work = n_tiles - g
    n_pad = -(-nq // 16) * 16
    kb = D // 128 if i8 else D // 64
    q_bytes = n_pad * 128 * (2 if i8 else 1)
    total = 0
    for c in range(g):
        tiles = 1 + len(range(c, n_work, g))        # the sample tile, then the round-robin share
        if i8 and i8_halves == 3:
            items = 1 + -(-(2 * (tiles - 1)) // 3)  # the sample tile's two halves alone, then the rest by three
            total += kb * (2 * tiles * 128 * 128 + items * q_bytes)
        else:
            total += kb * tiles * (TILE * 128 + q_bytes)
    return g, total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--i8-halves", type=int, choices=(2, 3), default=2,
                    help="128-row halves the int8 kernel stages per k-block of an item (2: one tile per item)")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    print("# %s -- name, power limit, SM clock, max SM clock, read in the same run" % smi())
    db32, q_host = bench.synthetic_inputs(torch, dev, 0, bench.N_DB, 0)
    index = Index.from_packed(pack_bf16(db32), db32=db32)
    index.stats()
    nq, D = bench.N_Q, bench.DIM
    kth = default_shortlist(bench.TOPK)
    route = index._route(kth, nq)
    assert route[0] == 1 and index._i8_route(kth, nq), "the bench shape must take the one-launch int8 route"
    q32 = q_host[0].to(dev)
    q8, _ = index._pack_q_i8(q32)
    q16 = pack_bf16(q32)
    launch = {"int8": lambda: index._first_pass(route, q8, kth, nq), "bf16": lambda: index._first_pass(route, q16, kth, nq)}
    hbm = {"int8": index.n * D + 4 * index.n, "bf16": index.n * D * 2}
    ingest = {"int8": fused_ingest(index.n, D, nq, True, args.i8_halves), "bf16": fused_ingest(index.n, D, nq, False, 0)}
    for f in launch.values():
        for _ in range(20):
            f()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = {k: [] for k in launch}
    for _ in range(ROUNDS):
        for k, f in launch.items():
            ev[0].record()
            for _ in range(REPS):
                f()
            ev[1].record()
            torch.cuda.synchronize()
            ms[k].append(ev[0].elapsed_time(ev[1]) / REPS)
    print("# after the timed rounds: %s" % smi())
    print("# bench data: %d rows x %d, %d queries, shortlist %d; CUDA events, mean of %d launches per round, %d rounds; "
          "int8 staged as %d halves per item" % (index.n, D, nq, kth, REPS, ROUNDS, args.i8_halves))
    for k in launch:
        g, ing = ingest[k]
        for t in ms[k]:
            print("%s fused scan: %.4f ms  HBM %.2f TB/s  ingest %.1f GB/s per SM (%d CTAs, %.2f ingest bytes per HBM byte)"
                  % (k, t, hbm[k] / (t * 1e-3) / 1e12, ing / (g * t * 1e-3) / 1e9, g, ing / hbm[k]))


if __name__ == "__main__":
    main()
