"""Anatomy of the certified finalize on the int8 route at the bench shape: two tiers (Index.tiered = False: the whole
extension gathered from the fp32 master) against three (the extension screened on the bf16 rows first).

bench.py's data (1,001,001 unit randn rows at D = 2048, 8 batches of 70 unit queries, top-100, the same seeds).  Per
batch, the int8 first pass runs once and both finalizes run on its output, so they see the same candidates.  Printed:
  - per query (over all batches): candidates, |S| (the shortlist), |E| (the extension: s8 >= t0 - eps8 outside S),
    |F| (rows of E with s16 >= t0 - eps16); counted on the host from the candidate list with fp64 scores, which can
    differ from the kernel's fp32 decisions only for rows within an ulp of a bound;
  - bytes gathered per step from db32 and db16 by each finalize;
  - finalize time by CUDA events (mean of REPS launches on one first-pass output, three alternating rounds);
  - eager Index.search (check=False) per step with each finalize (mean over 8 batches x 8 steps, three rounds);
  - whether the two finalizes return identical ids, scores and status words.
The card's name and power limit are read in the same run.

    python tools/time_finalize.py
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from mdir_b200.search import Index, pack_bf16, default_shortlist  # noqa: E402

REPS = 200


def key_scores(keys):
    """uint64 keys (numpy int64 view) -> fp32 scores (the inverse of make_key's desc_key)."""
    o = ~(keys.view(np.uint64) >> np.uint64(32)).astype(np.uint32)
    u = np.where(o >> np.uint32(31) != 0, o ^ np.uint32(0x80000000), o ^ np.uint32(0xffffffff)).astype(np.uint32)
    return u.view(np.float32)


def candidates(cand, cnt, caps, q):
    """The candidate keys of query q: the scan writes rows of cap0 + 148 * cap_l keys into the flat buffer."""
    cap0, cap_l = caps
    cand_row = cap0 + 148 * cap_l
    row, counts = cand.reshape(-1)[q * cand_row:(q + 1) * cand_row], cnt[q]
    parts = []
    for sg in range(counts.shape[0]):
        c = min(int(counts[sg]), cap0 if sg == 0 else cap_l)
        base = 0 if sg == 0 else cap0 + (sg - 1) * cap_l
        parts.append(row[base:base + c])
    return np.concatenate(parts)


def tiers(index, q32, cand, cnt, caps, q_eps, kth, k_out):
    """-> per query (n_cand, |S|, |E|, |F|) on the host."""
    st = index.stats().cpu().numpy().astype(np.float64)
    cand, cnt, q_eps = cand.cpu().numpy(), cnt.cpu().numpy().view(np.uint32), q_eps.cpu().numpy()
    D = index.D
    acc = 1.25 * D * 2.0 ** -24
    out = []
    for q in range(q32.shape[0]):
        keys = np.sort(candidates(cand, cnt, caps, q).view(np.uint64))
        s8 = key_scores(keys.view(np.int64)).astype(np.float64)
        slots = (keys & np.uint64(0xffffffff)).astype(np.int64) - index.idx_base
        assert keys.size and (slots >= 0).all() and (slots < index.n).all(), "candidate list decoded wrongly"
        nk = min(kth, keys.size)
        qd = q32[q].double()
        s32 = (index.db32[torch.from_numpy(slots[:nk]).to(q32.device)].double() @ qd).cpu().numpy()
        t0 = np.sort(s32)[::-1][k_out - 1]
        ext = np.flatnonzero((np.arange(keys.size) >= nk) & (s8 >= t0 - q_eps[q]))
        s16 = (index.db16[torch.from_numpy(slots[ext]).to(q32.device)].double() @ qd).cpu().numpy()
        qn = float(q32[q].double().norm())
        eps16 = (np.sqrt(st[0]) * qn + acc * (np.sqrt(st[1]) + np.sqrt(st[0])) * qn + acc * np.sqrt(st[1]) * qn) * 1.001 + 1e-7
        out.append((keys.size, nk, ext.size, int((s16 >= t0 - eps16).sum())))
    return np.array(out)


def main():
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout.strip()
    print("# %s -- the card of every number below, read in the same run" % smi)
    db32, q_host = bench.synthetic_inputs(torch, dev, 0, bench.N_DB, 0)
    q_bank = q_host.to(dev)
    index = Index.from_packed(pack_bf16(db32), db32=db32)
    index.stats()
    nq, k_out, D = bench.N_Q, bench.TOPK, bench.DIM
    kth = default_shortlist(k_out)
    route = index._route(kth, nq)
    assert route[0] == 1 and index._i8_route(kth, nq), "the bench shape must take the int8 route"
    out_s = {t: torch.empty((nq, k_out), dtype=torch.float32, device=dev) for t in (False, True)}
    out_i = {t: torch.empty((nq, k_out), dtype=torch.int32, device=dev) for t in (False, True)}
    ovf = {t: torch.empty((nq,), dtype=torch.int32, device=dev) for t in (False, True)}
    stats, same = [], True
    fin_ms = {False: [], True: []}
    for b in range(bench.N_BATCHES):
        q32 = q_bank[b]
        q8, q_eps = index._pack_q_i8(q32)
        tau, cand, cnt, caps = index._first_pass(route, q8, kth, nq)
        tau, cand, cnt, q_eps = tau.clone(), cand.clone(), cnt.clone(), q_eps.clone()

        def fin(t):
            index.tiered = t
            index._finalize(cand, cnt, nq, kth, out_s[t], out_i[t], None, tau, ovf[t], (q32, k_out), caps, q_eps)

        for t in (False, True):
            fin(t)
        torch.cuda.synchronize()
        same &= bool(torch.equal(out_s[False], out_s[True]) and torch.equal(out_i[False], out_i[True]) and torch.equal(ovf[False], ovf[True]))
        stats.append(tiers(index, q32, cand, cnt, caps, q_eps, kth, k_out))
        if b == 0:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            for _ in range(3):
                for t in (False, True):
                    fin(t)
                    ev[0].record()
                    for _ in range(REPS):
                        fin(t)
                    ev[1].record()
                    torch.cuda.synchronize()
                    fin_ms[t].append(ev[0].elapsed_time(ev[1]) / REPS)
    index.tiered = True
    st = np.concatenate(stats)
    print("# bench data: %d rows x %d, %d batches x %d queries, top-%d, shortlist %d, int8 route" % (index.n, D, bench.N_BATCHES, nq, k_out, kth))
    for j, name in enumerate(("candidates", "|S|", "|E|", "|F|")):
        print("%-10s per query: mean %7.1f  min %5d  max %5d" % (name, st[:, j].mean(), st[:, j].min(), st[:, j].max()))
    s_, e_, f_ = st[:, 1].mean() * nq, st[:, 2].mean() * nq, st[:, 3].mean() * nq
    print("gathered per step, two tiers:   db32 %.3f GB" % ((s_ + e_) * D * 4 / 1e9))
    print("gathered per step, three tiers: db32 %.3f GB + db16 %.3f GB" % ((s_ + f_) * D * 4 / 1e9, e_ * D * 2 / 1e9))
    print("identical ids, scores and status words (8 batches): %s" % same)
    for t, name in ((False, "two tiers  "), (True, "three tiers")):
        print("finalize %s: %s ms (CUDA events, mean of %d launches, 3 rounds)" % (name, " ".join("%.4f" % v for v in fin_ms[t]), REPS))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    step_ms = {False: [], True: []}
    for _ in range(3):
        for t in (False, True):
            index.tiered = t
            for b in range(bench.N_BATCHES):
                index.search(q_bank[b], k_out, precision="fp32", check=False)
            torch.cuda.synchronize()
            ev[0].record()
            for _ in range(8):
                for b in range(bench.N_BATCHES):
                    index.search(q_bank[b], k_out, precision="fp32", check=False)
            ev[1].record()
            torch.cuda.synchronize()
            step_ms[t].append(ev[0].elapsed_time(ev[1]) / (8 * bench.N_BATCHES))
    index.tiered = True
    for t, name in ((False, "two tiers  "), (True, "three tiers")):
        print("eager search step %s: %s ms (check=False, 64 steps, 3 rounds)" % (name, " ".join("%.4f" % v for v in step_ms[t])))


if __name__ == "__main__":
    main()
