#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric on its own configuration:

    queries/s against a 1,001,001 x 2048 database (R1M shape, config 4), 70 queries per step,
    top-100 per query identical to the fp32 reference ranking (bf16 tcgen05 scan + fused
    threshold filter + exact fp32 re-scoring of a 132-entry shortlist),
    on N B200s of one node (database rows sharded, local top-k, one NCCL all-gather of keys).

A "step" = one batch of 70 queries ranked against the whole database.
  value  : device-resident queries, CUDA-event timed, max over ranks
  e2e    : the same through the public API with HOST buffers: pinned-host queries -> H2D ->
           search -> D2H of the (scores, idx) result, every step.  The database is the resident
           index (state, like weights), not a per-step input; `e2e_cold_db_ms` reports the
           one-off upload + bf16 packing of the database separately.
  --impl reference : the reference's CPU path (np.dot + np.argsort, cirscore.py:69-70, restated
           in oracle/oracle.py) on the host cores, on a bounded row sample of the same workload.

Launch: python bench.py [--gpus N --steps K --warmup W]; for N > 1 under torchrun
(python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...).
--dump-outputs DIR writes the result of the last timed step (DIR/scores.npy, DIR/indices.npy).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_DB, DIM, N_Q, TOPK = 1001001, 2048, 70, 100
METRIC = "queries/s vs 1M x 2048 db (70-query batches, top-100, fp32-faithful ranking)"
UNIT = "queries/s"
WORKLOAD = "R1M: 70 q x 1,001,001 x 2048-D db, top-100 (BASELINE.json configs[3]; 4.1 GB bf16 + 8.2 GB fp32 master)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the head / CLAHE / C5 side measurements")
    ap.add_argument("--full-dba", action="store_true", help="N=1: run the full 1M-row DBA instead of a 16,384-row slice")
    ap.add_argument("--cpu-rows", type=int, default=200000, help="database row sample for the cpu_baseline leg of our arm")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the (scores, indices) of the last timed step to DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


def dump_outputs(path, scores, idx):
    """The result a caller of the timed step receives: top-k scores (float32) and database row indices (float64, exact
    for every row index), both (queries, k), best first.  The inputs are seeded, so two builds can be compared file by file."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "scores.npy"), scores.cpu().numpy().astype(np.float32))
    np.save(os.path.join(path, "indices.npy"), idx.cpu().numpy().astype(np.float64))


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------ CPU reference arm
REF_BUDGET_S = 210.0      # wall-clock budget of the whole --impl reference run (data generation excluded)


def host_cores():
    return len(os.sched_getaffinity(0))


def host_descriptors(rows, seed, threads):
    """(D, rows) fp32 C-order with unit columns -- the layout extract_vectors returns (imageretrievalnet.py:291) --
    filled by `threads` numpy Generators in parallel (they release the GIL)."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    vecs = np.empty((DIM, rows), dtype=np.float32)
    step = max(4096, -(-rows // (4 * threads)))

    def fill(c0):
        c1 = min(rows, c0 + step)
        blk = np.random.default_rng([seed, c0]).standard_normal((DIM, c1 - c0), dtype=np.float32)
        blk /= np.sqrt((blk * blk).sum(axis=0, keepdims=True))
        vecs[:, c0:c1] = blk
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(fill, range(0, rows, step)))
    return vecs


def reference_step(vecs, qvecs):
    """Exactly what cirscore.py:69-70 executes (restated in oracle/oracle.py:scores): np.dot(vecs.T, qvecs) and
    np.argsort(-scores, axis=0) with numpy's default sort kind."""
    import numpy as np
    from oracle import oracle
    sc = oracle.scores(vecs, qvecs)
    return np.argsort(-sc, axis=0)


def time_reference(vecs, qvecs, steps, warmup, threads):
    """-> list of per-step seconds, BLAS pinned to `threads` whatever OMP_NUM_THREADS says (torchrun sets it to 1)."""
    from threadpoolctl import threadpool_limits
    ts = []
    with threadpool_limits(limits=threads):
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            rk = reference_step(vecs, qvecs)
            dt = time.perf_counter() - t0
            assert rk.shape == (vecs.shape[1], qvecs.shape[1])
            if i >= warmup:
                ts.append(dt)
    return ts


def cpu_reference(rows, reps, threads=None, vecs=None, qvecs=None):
    """The reference arithmetic on `rows` database rows x 70 queries, `threads` BLAS threads (default: every host core);
    queries/s scaled linearly to the full database when rows < N_DB (argsort is n log n, so that flatters the CPU)."""
    import numpy as np
    threads = threads or host_cores()
    if vecs is None:
        vecs = host_descriptors(rows, 4, host_cores())
        qvecs = host_descriptors(N_Q, 5, 1)
    ts = time_reference(vecs[:, :rows], qvecs, reps, 1, threads)
    t = float(np.median(ts))
    scale = N_DB / float(rows)
    return {"value": N_Q / (t * scale), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "np.dot + np.argsort(axis=0) (cirscore.py:69-70 via the oracle port) on %d of %d db rows x 70 queries x 2048-D, %d BLAS threads of %d host cores, median of %d%s"
                      % (rows, N_DB, threads, host_cores(), reps, "" if rows == N_DB else ", time scaled x%.2f" % scale),
            "ms_per_step": t * scale * 1e3, "rows": rows}


def run_reference(args):
    """bench.py --impl reference: the reference's own CPU implementation of the path on this box's host cores, at the
    FULL workload (1,001,001 rows per step) for --warmup + --steps steps when that fits REF_BUDGET_S; otherwise the
    steps run on the largest row sample that does, after one full-size step, and the line says so."""
    import numpy as np
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    t_gen = time.perf_counter()
    vecs = host_descriptors(N_DB, 4, cores)
    qvecs = host_descriptors(N_Q, 5, 1)
    t_gen = time.perf_counter() - t_gen
    t_start = time.perf_counter()
    full = time_reference(vecs, qvecs, 1, 0, cores)[0]                     # one full-size step, always (also the first warm-up)
    warm = max(args.warmup, 1)
    total_steps = warm - 1 + args.steps
    rows = N_DB
    if total_steps * full > REF_BUDGET_S - full:
        rows = int(max(50000, min(N_DB, N_DB * (REF_BUDGET_S - full) / (total_steps * full))))
    ts = time_reference(vecs[:, :rows] if rows < N_DB else vecs, qvecs, args.steps, warm - 1, cores)
    scale = N_DB / float(rows)
    t = float(np.mean(ts)) * scale
    # the as-shipped thread setting of the reference (torch/MKL/OMP = 3, mdir/stages/validate.py:10-12), for the record
    t3 = None
    if time.perf_counter() - t_start < REF_BUDGET_S:
        r3 = min(rows, 250000)
        t3 = float(np.median(time_reference(vecs[:, :r3], qvecs, 2, 1, 3))) * (N_DB / float(r3))
    sample = ("every step = the full workload: np.dot(vecs.T, qvecs) + np.argsort(-scores, axis=0) (cirscore.py:69-70 via the oracle port) on "
              "1,001,001 x 2048 fp32 x 70 queries" if rows == N_DB else
              "steps on %d of %d db rows (time scaled x%.2f) to fit %.0f s; one full-size step took %.0f ms" % (rows, N_DB, scale, REF_BUDGET_S, full * 1e3))
    sample += "; %d BLAS threads (all host cores, pinned with threadpoolctl regardless of OMP_NUM_THREADS)" % cores
    line = {"impl": "reference", "metric": METRIC, "value": N_Q / t, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": warm, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD},
            "cpu_baseline": {"value": N_Q / t, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": N_Q / t, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "full_size_step_ms": full * 1e3, "rows_per_step": rows, "host_data_generation_s": t_gen,
            "as_shipped_3_threads": None if t3 is None else {"value": N_Q / t3, "unit": UNIT, "ms_per_step": t3 * 1e3, "cores": 3,
                                                              "note": "torch/MKL/OMP = 3 threads as mdir/stages/validate.py:10-12 sets them; 250k-row sample scaled"}}
    print(json.dumps(line))


# ------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, torch_device_index):
        super().__init__(daemon=True)
        self.samples = []
        self.stop_flag = False
        self.active = False
        self.ok = False
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            uuid = str(torch.cuda.get_device_properties(torch_device_index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(torch_device_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as exc:  # noqa: BLE001
            self.err = repr(exc)

    def run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((self.active, mhz, reasons))
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": getattr(self, "err", "nvml unavailable")}
        import statistics
        act = [s for s in self.samples if s[0]] or self.samples
        names = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
                 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        bits = 0
        for _, _, r in act:
            bits |= r
        return {"sm_mhz": statistics.median([s[1] for s in act]) if act else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for b, n in names.items() if bits & b and n != "gpu_idle"), "samples": len(act)}


class KernelProf:
    """One pair of CUDA events around the dominant kernel, on the stream it is launched on.  The
    events are `external` so that they become record nodes when the step is captured into a CUDA
    graph: after a replay + synchronize, elapsed_time() is that replay's kernel duration."""

    def __init__(self, torch):
        self.e0 = torch.cuda.Event(enable_timing=True, external=True)
        self.e1 = torch.cuda.Event(enable_timing=True, external=True)
        self.bytes = 0

    def begin(self):
        self.e0.record()

    def end(self, nbytes):
        self.e1.record()
        self.bytes = nbytes

    def last_ms(self):
        return self.e0.elapsed_time(self.e1)


class QuietStdout:
    """Everything libraries print to fd 1 while the benchmark runs (NCCL's version banner, ...) goes to stderr, so
    that stdout carries exactly one line: the JSON result written through emit()."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.real, (text + "\n").encode())


# ------------------------------------------------------------------ our arm
def count_launches_per_step(lib, target, q_dev):
    """Kernels of libmdir_b200 launched by one step (counted on an un-captured run of the same call)."""
    n0 = lib.mdir_launch_count()
    target.search(q_dev, TOPK, precision="fp32", check=False)
    return int(lib.mdir_launch_count() - n0)


N_BATCHES = 8             # distinct query batches rotated through every timed loop


def same_topk(got_i, got_s, ref_i, ref_v, tol):
    """got (nq, k) vs an independent reference ranking ref (nq, k_ext >= k): scores equal to tol position by position,
    every index mismatch must be a swap inside a reference gap <= tol.  -> (violations, swaps_inside_gaps)."""
    import numpy as np
    nq, k = got_i.shape
    bad = int((np.abs(got_s - ref_v[:, :k]) > tol).sum())
    swaps = 0
    for j in range(nq):
        for r in np.nonzero(got_i[j] != ref_i[j, :k])[0]:
            near = np.abs(ref_v[j] - ref_v[j, r]) <= tol
            if got_i[j, r] in ref_i[j][near]:
                swaps += 1
            else:
                bad += 1
    return bad, swaps


def independent_topk(torch, mdir_b200, index, q, k_ext):
    """Local top-k_ext of one shard by a path that shares nothing with the bf16 shortlist machinery: dense 3xTF32 scores
    of every row -> exact select -> fp64 re-scoring by torch.  -> (global idx (nq, k_ext + 48) int64, fp64 scores) unsorted-by-fp64."""
    dense = index.scores(q, precision="fp32")
    idx, _ = mdir_b200.topk_from_scores(dense.t().contiguous(), min(k_ext + 48, index.n))
    del dense
    idx = idx.t().contiguous()
    v64 = (index.db32[idx.reshape(-1)].double().view(idx.shape[0], idx.shape[1], -1) * q.double()[:, None, :]).sum(-1)
    return idx + index.idx_base, v64


def synthetic_inputs(torch, dev, lo, hi, rank):
    """The seeded inputs of our arm: database shard rows [lo, hi) of the 1,001,001 (unit fp32 rows, built on `dev`)
    and the N_BATCHES query batches (N_BATCHES, N_Q, DIM) on the host."""
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    db32 = torch.empty((hi - lo, DIM), dtype=torch.float32, device=dev)
    for r0 in range(0, hi - lo, 65536):
        blk = torch.randn((min(65536, hi - lo - r0), DIM), device=dev, generator=g)
        db32[r0:r0 + blk.shape[0]] = blk / blk.norm(dim=1, keepdim=True)
    gq = torch.Generator(device="cpu").manual_seed(99)
    q = torch.randn((N_BATCHES, N_Q, DIM), generator=gq)
    return db32, q / q.norm(dim=2, keepdim=True)


def run_ours(args):
    import numpy as np
    import torch
    import mdir_b200
    from mdir_b200 import _lib
    from mdir_b200.search import Index, ShardedIndex, GraphedSearch, SearchPipeline, pack_bf16, default_shortlist

    out = QuietStdout()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun (python -m torch.distributed.run --nproc-per-node %d bench.py ...)" % (args.gpus, args.gpus))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    _lib.check(_lib.lib().mdir_device_check(), "device check")
    lib = _lib.lib()

    lo, hi = ShardedIndex.shard_bounds(N_DB, world, rank)
    db32, q_host = synthetic_inputs(torch, dev, lo, hi, rank)
    q_host = q_host.pin_memory()                                      # every timed loop rotates through these batches
    q_bank = q_host.to(dev)
    torch.cuda.synchronize()
    # cold path of the index build (packing only; the fp32 rows are already resident)
    t0 = time.perf_counter()
    index = Index.from_packed(pack_bf16(db32), db32=db32, idx_base=lo)
    index.stats()                                                    # database half of the shortlist certificate (one pass, cached)
    torch.cuda.synchronize()
    pack_ms = (time.perf_counter() - t0) * 1e3
    prof = KernelProf(torch)
    target = ShardedIndex.from_local(index) if world > 1 else index
    # the whole step (pack q, fused threshold+filter scan, finalize + certified fp32 re-score, [exchange + merge]) captured
    # once per query batch into a CUDA graph whose static query buffer already holds that batch: every timed step is ONE
    # graph replay, and consecutive steps search different queries
    # N > 1: one graph holds pack + scan, a second one finalize + certified re-score; the second graph and the NVLink
    # push + merge of step t are launched on a second stream and run while step t+1 scans (GraphedSearch(overlap=True,
    # split=True)); every step's merged result is produced, none skipped
    # N = 1: one graph per step (the split was measured there too -- tools/time_split_1gpu.py: 660 us as one graph,
    # 664-705 us split: capping the scan grid costs what hiding finalize gains)
    deferred = False
    graphs = []
    for b in range(N_BATCHES):
        gb = GraphedSearch(target, N_Q, TOPK, precision="fp32", overlap=(world > 1 and getattr(target, "_mb", None) is not None), split=True)
        gb.q.copy_(q_bank[b])
        gb.used = False
        graphs.append(gb)
    overlap = all(gb.overlap for gb in graphs)
    exch_stream = torch.cuda.Stream(device=dev) if overlap else None
    gs = GraphedSearch(target, N_Q, TOPK, precision="fp32")          # synchronous exchange: the blocking e2e loop
    # the same step with a CUDA event pair around the dominant kernel inside the graph: used only to read that
    # kernel's duration (the two event-record nodes cost ~8 us per step, so `value` is timed on the plain graphs)
    gs_prof = GraphedSearch(target, N_Q, TOPK, precision="fp32", prof=prof)
    gs_prof.q.copy_(q_bank[0])
    out_host = torch.empty((N_Q, TOPK * 2), dtype=torch.float32).pin_memory()

    def step_e2e(t):
        s, i = gs(q_host[t % N_BATCHES])                             # pinned host -> static device buffer, replay
        out_host[:, :TOPK].copy_(s, non_blocking=True)
        out_host[:, TOPK:].view(torch.int32).copy_(i, non_blocking=True)
        torch.cuda.synchronize()
        return out_host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(n):
        cur = torch.cuda.current_stream(dev)
        for t in range(n):
            gb = graphs[t % N_BATCHES]
            if not overlap:
                gb.graph.replay()
                continue
            if gb.used:
                cur.wait_event(gb.done)                    # the previous exchange of this graph has read its key buffer
            gb.graph.replay()
            gb.local_done.record(cur)
            with torch.cuda.stream(exch_stream):
                exch_stream.wait_event(gb.local_done)
                gb.exchange()
                gb.done.record(exch_stream)
            gb.used = True
        if overlap:
            cur.wait_stream(exch_stream)                   # the timed region ends when the last step's merge is done

    # ---- warm-up ---------------------------------------------------------------------------------
    run_steps(max(args.warmup, 3))
    torch.cuda.synchronize()
    for t in range(3):
        step_e2e(t)

    # ---- timed region: `value` ------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if sampler.ok:
        sampler.start()
    n0 = lib.mdir_launch_count()
    target.search(q_bank[0], TOPK, precision="fp32", check=False)
    launches_per_step = int(lib.mdir_launch_count() - n0)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    sampler.active = True
    ev[0].record()
    run_steps(args.steps)
    ev[1].record()
    barrier()
    sampler.active = False
    launches = launches_per_step * args.steps
    ms_total = ev[0].elapsed_time(ev[1])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *graphs[(args.steps - 1) % N_BATCHES].out)
    # dominant-kernel duration: the graph carries an event pair around the scan; read it after individual replays
    # of the same graph (a per-step read needs a sync, so not inside the loop above)
    scan_samples = []
    for _ in range(min(50, args.steps) + 1):
        gs_prof()
        torch.cuda.synchronize()
        scan_samples.append(prof.last_ms())
    scan_ms = sum(scan_samples) / len(scan_samples)

    # ---- timed region: e2e (host buffers in, host result out, every step) --------------------------
    # (1) blocking: upload, replay, download, synchronize -- the latency of one step seen from the host
    barrier()
    t0 = time.perf_counter()
    for t in range(args.steps):
        step_e2e(t)
    barrier()
    e2e_blocking_s = time.perf_counter() - t0
    # (2) the serving loop (SearchPipeline): the same three stages per step, several steps in flight, so the copies of
    # one step overlap the scan of the next.  Every step's queries are uploaded and every result is read on the host.
    pipe = SearchPipeline(target, N_Q, TOPK, precision="fp32")
    for _ in pipe.map(q_host[b] for b in range(4)):
        pass
    barrier()
    t0 = time.perf_counter()
    n_out = 0
    for s_h, i_h in pipe.map(q_host[t % N_BATCHES] for t in range(args.steps)):
        n_out += int(i_h[0, 0] >= 0)
    barrier()
    e2e_s = time.perf_counter() - t0
    assert n_out == args.steps
    sampler.stop_flag = True

    # bf16-only mode (no fp32 re-scoring), for the record
    gs16 = GraphedSearch(target, N_Q, TOPK, precision="bf16")
    gs16.q.copy_(q_bank[0])
    for _ in range(3):
        gs16()
    e2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    e2[0].record()
    n_b = max(10, args.steps // 4)
    for _ in range(n_b):
        gs16()
    e2[1].record()
    torch.cuda.synchronize()
    bf16_ms = e2[0].elapsed_time(e2[1]) / n_b

    per_rank = None
    if world > 1:
        mine = torch.tensor([ms_total, e2e_s, scan_ms], dtype=torch.float64, device=dev)
        allr = torch.empty((world, 3), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allr.view(-1), mine)
        per_rank = {"ms_total": allr[:, 0].tolist(), "e2e_s": allr[:, 1].tolist(), "scan_ms": allr[:, 2].tolist()}
        ms_total, e2e_s, scan_ms = [float(x) for x in allr.max(dim=0).values.tolist()]

    # ---- parity of what was timed (VERDICT r1 items 1-2) -------------------------------------------------
    # For every one of the N_BATCHES query batches: the result of the TIMED graph (at N > 1: local certified top-k,
    # keys pushed over NVLink, merge deferred by a step) against (a) an independent ranking -- per shard dense 3xTF32
    # scores of every row -> exact select -> fp64 re-scoring, shards merged on the host -- with swaps accepted only
    # inside 2e-6 reference gaps, and at N > 1 (b) bit for bit against the ncclAllGather + merge-kernel route.
    K_EXT = TOPK + 16
    timed, flagged = [], 0
    for b in range(N_BATCHES):
        graphs[b]()                                        # replay (+ this step's exchange and merge at N > 1)
        torch.cuda.synchronize()
        timed.append((graphs[b].out[0].clone(), graphs[b].out[1].clone()))
        flagged += int(graphs[b].status.ne(0).sum().item())
    nccl_equal = None
    if world > 1:
        ShardedIndex.p2p = False
        nccl_index = ShardedIndex.from_local(index)
        ShardedIndex.p2p = True
        nccl_equal = True
        for b in range(N_BATCHES):
            s_n, i_n = nccl_index.search(q_bank[b], TOPK, precision="fp32")
            nccl_equal &= bool(torch.equal(i_n, timed[b][1]) and torch.equal(s_n, timed[b][0]))
    violations = swaps = 0
    for b in range(N_BATCHES):
        r_i, r_v = independent_topk(torch, mdir_b200, index, q_bank[b], K_EXT)
        if world > 1:
            g_i = torch.empty((world,) + tuple(r_i.shape), dtype=r_i.dtype, device=dev)
            g_v = torch.empty((world,) + tuple(r_v.shape), dtype=r_v.dtype, device=dev)
            dist.all_gather_into_tensor(g_i.view(-1), r_i.contiguous().view(-1))
            dist.all_gather_into_tensor(g_v.view(-1), r_v.contiguous().view(-1))
            r_i = g_i.permute(1, 0, 2).reshape(N_Q, -1)
            r_v = g_v.permute(1, 0, 2).reshape(N_Q, -1)
        r_i, r_v = r_i.cpu().numpy(), r_v.cpu().numpy()
        order = np.lexsort((r_i, -r_v), axis=1)[:, :K_EXT]
        r_i, r_v = np.take_along_axis(r_i, order, 1), np.take_along_axis(r_v, order, 1)
        bad, sw = same_topk(timed[b][1].cpu().numpy().astype(np.int64), timed[b][0].cpu().numpy().astype(np.float64), r_i, r_v, 2e-6)
        violations += bad
        swaps += sw
    index._db_x3 = None                                              # 24.6 GB / world of 3xTF32 operands: only the check needed them
    torch.cuda.empty_cache()
    parity = {"checked_queries": N_BATCHES * N_Q, "mismatches": violations, "swaps_inside_2e-6_reference_gaps": swaps,
              "certificate_failures": flagged, "certificate_counters": dict(index.cert),
              "reference": "independent: per shard dense 3xTF32 scores of every row -> exact top-%d select -> fp64 re-scoring (torch), shards merged on the host" % (K_EXT + 48),
              "timed_route": (("CUDA graph of pack + scan; finalize graph%s on a second stream" % (" + NVLink exchange/merge kernel" if world > 1 else "")) if overlap else "CUDA graph") + ", %d distinct query batches" % N_BATCHES}
    if nccl_equal is not None:
        parity["p2p_route_equals_nccl_allgather_route"] = nccl_equal
        flag = torch.tensor([violations, 0 if nccl_equal else 1], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)                                    # every rank merged the same lists
        parity["mismatches_max_over_ranks"], parity["p2p_route_equals_nccl_allgather_route"] = int(flag[0].item()), not bool(flag[1].item())
    assert parity["mismatches"] == 0, parity

    extras = {}
    if not args.no_extras:
        extras.update(c5_measurements(torch, dist, world, rank, target, index, q_bank[0], args))
    if rank == 0 and not args.no_extras:
        if world == 1:
            extras.update(search_side_measurements(torch, mdir_b200, index, q_bank[0], prof))
        extras.update(side_measurements(torch, mdir_b200, dev))

    if rank != 0:
        finish(dist, world)
        return

    peak, peak_src = measured_peaks()
    achieved = prof.bytes / 1e9 / (scan_ms * 1e-3) if scan_ms > 0 else None
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "sim_scan_traffic.json")
    if os.path.exists(tpath) and world == 1:      # the ncu capture is of the 1-GPU launch
        with open(tpath) as fh:
            traffic = json.load(fh).get("dram_bytes_per_launch")
    ms_step = ms_total / args.steps
    line = {
        "metric": METRIC, "value": N_Q * args.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "queries_per_step": N_Q, "topk": TOPK, "shortlist": default_shortlist(TOPK),
                   "distinct_query_batches": N_BATCHES, "db_rows_per_gpu": hi - lo,
                   "pipeline": ("step = CUDA graph {pack, scan} on the compute stream + CUDA graph {finalize, certified re-score}%s on a second stream, "
                                "overlapping the next step's scan%s" % (" + exchange/merge kernel" if world > 1 else "", ""))
                               if overlap else "one CUDA graph per step",
                   "sharding": "db rows contiguous over %d GPU(s); %s" % (world, "single shard" if world == 1 else (
                       ("%d B of keys per rank pushed to every peer over NVLink by the merge kernel itself (no NCCL call on the step); finalize, exchange and "
                        "merge of step t run on a second stream while step t+1 scans") % (N_Q * TOPK * 8) if overlap else
                       "ncclAllGather of %d B of keys per rank + merge kernel" % (N_Q * TOPK * 8))),
                   "l2": "inputs larger than L2: %.2f GB bf16 shard streamed per step vs 126 MB L2" % ((hi - lo) * DIM * 2 / 1e9)},
        "clocks": sampler.summary(),
        "e2e": {"value": N_Q * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": N_Q * DIM * 4, "d2h_bytes_per_step": N_Q * TOPK * 8 + N_Q * 4,
                "ms_per_step": e2e_s / args.steps * 1e3, "blocking_ms_per_step": e2e_blocking_s / args.steps * 1e3, "steps_redone_exactly": pipe.n_recovered,
                "timing": "wall clock around %d steps of SearchPipeline (per step: H2D of the pinned queries, graph replay, D2H of scores/idx/status, host read of the result; %d steps in flight%s); blocking_ms_per_step = the same with a synchronize after every step" % (args.steps, pipe.depth, ", NVLink exchange overlapped with the next scan" if pipe.overlap else "")},
        "e2e_cold_db_ms": {"pack_fp32_to_bf16_and_certificate_stats_ms": pack_ms,
                           "note": "one-off index build for this shard; host->device upload of the fp32 rows would add %.1f GB over PCIe" % ((hi - lo) * DIM * 4 / 1e9)},
        "gpu_launches": int(launches), "gpu_launches_note": "%d libmdir_b200 kernels per step, replayed from one CUDA graph per step" % launches_per_step,
        "roofline": {"bound": "hbm", "kernel": "sim_scan_kernel (%s)" % ("threshold + filter in one launch: whole shard" if index._fused_ok(default_shortlist(TOPK)) else "FILTER pass"), "achieved": achieved, "peak": peak, "peak_source": peak_src,
                     "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                     "algorithmic_bytes_per_launch": prof.bytes, "avg_launch_ms": scan_ms, "share_of_step": scan_ms / ms_step,
                     "timing": "CUDA events (external, recorded inside the step's CUDA graph on its stream), mean of %d replays" % len(scan_samples)},
        "parity_check": parity,
        "bf16_only_ms_per_step": bf16_ms,
    }
    if world == 1:
        cb = cpu_reference(args.cpu_rows, 3)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        cb3 = cpu_reference(min(args.cpu_rows, 100000), 2, threads=3)
        line["cpu_baseline_as_shipped_3_threads"] = {k: cb3[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if per_rank is not None:
        line["per_rank"] = per_rank
    line.update(extras)
    out.emit(json.dumps(line))
    sys.stdout.flush()
    finish(dist, world)


def c5_measurements(torch, dist, world, rank, target, index, q_dev, args):
    """BASELINE.json configs[4] (alpha-QE + DBA on the 1M x 2048 database) at THIS world size; every rank takes part.
    alpha-QE: search top-10, expand (one all-reduce of N_q x D fp32 when sharded), search top-100.
    DBA: every database row searched against the whole database (top-10) and replaced by the weighted sum of its
    neighbours.  Run in full at N > 1 (the verdict's 8-GPU measurement); at N = 1 a bounded 16,384-row slice of the
    database rows is augmented and the full run extrapolated linearly (a full pass is seconds; --full-dba runs it)."""
    from mdir_b200 import qe
    out = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_ms(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=q_dev.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(2):
        qe.search_qe(target, q_dev, TOPK)
    barrier()
    ev[0].record()
    for _ in range(10):
        qe.search_qe(target, q_dev, TOPK)
    ev[1].record()
    barrier()
    ms = max_ms(ev[0].elapsed_time(ev[1]) / 10)
    out["alpha_qe"] = {"metric": "alpha-QE queries/s (alpha=3, n_QE=10; two certified similarity+top-k passes%s; parity unpinned)" % (
                           "" if world == 1 else " + one all-reduce of the expansion"),
                       "value": N_Q / (ms * 1e-3), "unit": "queries/s", "ms_per_batch": ms, "n_gpus": world}
    full = world > 1 or args.full_dba
    if not full:
        qe.dba(index, 3.0, 10, rows=4096)                # warm: the wide candidate / sample workspaces are allocated on first use
    barrier()
    t0 = time.perf_counter()
    if full:
        aug = qe.dba_sharded(target, 3.0, 10) if world > 1 else qe.dba(index, 3.0, 10)
        rows_done = N_DB
    else:
        rows_done = 16384
        aug = qe.dba(index, 3.0, 10, rows=rows_done)
    barrier()
    dba_s = max_ms((time.perf_counter() - t0) * 1e3) / 1e3
    del aug
    torch.cuda.empty_cache()
    flops = 2.0 * rows_done * N_DB * DIM
    out["dba"] = {"metric": "DBA (k=10, alpha=3) over the 1,001,001 x 2048 database, every row searched against every row",
                  "n_gpus": world, "rows_augmented": rows_done, "seconds": dba_s,
                  "full_1M_seconds": dba_s * (N_DB / rows_done), "measured_in_full": bool(full),
                  "tflops_per_gpu": flops / dba_s / 1e12 / world,
                  "note": "wall clock incl. the all-gather of the shards, index build and per-block host loop; max over ranks"}
    return out


def finish(dist, world):
    """Multi-rank exit: barrier, then leave without tearing NCCL down (communicators referenced by
    captured CUDA graphs make destroy_process_group() block)."""
    if world > 1:
        import torch
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def search_side_measurements(torch, mdir_b200, index, q_dev, prof):
    """The tensor-utilisation evidence on the resident 1M x 2048 index (1 GPU): blocks of 128 database rows searched
    against the whole database (the DBA inner loop), the 128-query FILTER scan as TFLOP/s."""
    out = {}
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    tf_peak = 1397.3
    if os.path.exists(path):
        with open(path) as fh:
            tf_peak = float(json.load(fh).get("bf16_tflops_sustained", tf_peak))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    # 1,024-row blocks of the database as queries (the DBA inner loop): ONE wide FILTER launch per block, work items =
    # (256-row tile, 128-query block): the tile comes from HBM once and from L2 seven times -> tensor-bound
    BLK = 1024
    rows = index.db32[:10 * BLK]
    index.prof = prof
    index.search(rows[:BLK], 10, precision="bf16", block_q=BLK)
    torch.cuda.synchronize()
    scan = []
    ev[0].record()
    for b in range(10):
        index.search(rows[b * BLK:(b + 1) * BLK], 10, precision="bf16", check=False, block_q=BLK)
        torch.cuda.synchronize()
        scan.append(prof.last_ms())
    ev[1].record()
    torch.cuda.synchronize()
    flagged = bool(index.check_overflow())
    index.prof = None
    ms_blk = ev[0].elapsed_time(ev[1]) / 10
    scan_ms = sum(scan) / len(scan)
    flops = 2.0 * BLK * DIM * (prof.bytes / (2 * DIM))
    out["dba_block"] = {"metric": "DBA inner loop: 1,024 database rows vs 1,001,001 x 2048 (top-10, bf16 scores), one wide launch per block", "ms_per_block": ms_blk,
                        "rows_per_s": BLK / (ms_blk * 1e-3), "full_dba_1M_estimate_s": (N_DB / float(BLK)) * ms_blk * 1e-3,
                        "block_tflops_incl_sample_select_finalize": 2.0 * BLK * DIM * N_DB / (ms_blk * 1e-3) / 1e12,
                        "filter_scan_ms": scan_ms, "filter_scan_tflops": flops / (scan_ms * 1e-3) / 1e12,
                        "frac_of_sustained_bf16_peak": flops / (scan_ms * 1e-3) / 1e12 / tf_peak, "bf16_peak_tflops_sustained": tf_peak,
                        "flagged": flagged,
                        "note": "8 query blocks per database tile: AI = 1,024 FLOP per HBM byte (ridge ~214); was 128 queries per pass, HBM-bound at 0.43-0.52 of the tensor peak"}
    return out


def side_measurements(torch, mdir_b200, dev):
    """The second half of BASELINE.json's metric: GeM + whiten descriptors/s (C2 head shape) and
    CLAHE images/s, each with its HBM-roofline fraction.  Outside the timed region of `value`."""
    from mdir_b200 import _lib
    peak, _ = measured_peaks()
    out = {}
    # head: 192 images x 3 scales of 2048 x {32x24, 23x17, 16x12}; P 2048x2048
    B, C = 192, 2048
    hws = [(32, 24), (23, 17), (16, 12)]
    g = torch.Generator(device=dev).manual_seed(7)
    fm = []
    for _ in range(B):
        for (h, w) in hws:
            fm.append(torch.randn((1, C, h, w), device=dev, generator=g).clamp_(min=0))
    P = torch.randn((C, C), device=dev, generator=g) / C ** 0.5
    m = torch.randn((C, 1), device=dev, generator=g) * 0.01
    head = mdir_b200.RetrievalHead("gem", p=2.9137, whitening={"P": P.cpu().numpy(), "m": m.cpu().numpy()}, nscales=3, device=dev)
    packed = head.pack(fm)                 # offset tables built once (static shapes), maps stay where they are
    for _ in range(3):
        head(packed)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    reps = 10
    for _ in range(reps):
        head(packed)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / reps
    bytes_img = 4 * C * sum(h * w for h, w in hws)
    replay = head.capture(packed)          # the same launches recorded once into a CUDA graph (static arena)
    for _ in range(3):
        replay()
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(reps):
        replay()
    ev[1].record()
    torch.cuda.synchronize()
    ms_g = ev[0].elapsed_time(ev[1]) / reps
    out["head"] = {"metric": "GeM+L2N+multiscale+Lw descriptors/s (C2 head: 3 scales, 2048-D)", "value": B / (ms_g * 1e-3), "unit": "descriptors/s",
                   "batch": B, "ms_per_batch": ms_g, "ms_per_batch_eager_launches": ms, "algorithmic_bytes_per_descriptor": bytes_img,
                   "hbm_frac_of_measured": B * bytes_img / 1e9 / (ms_g * 1e-3) / peak,
                   "note": "value = CUDA-graph replay of the head over a static feature-map arena; ms_per_batch_eager_launches = the same nine launches issued one by one"}
    del fm
    # CLAHE: 256 images of 768 x 1024 u8 (night-like gamma distribution)
    n_img = 256
    imgs = (torch.rand((n_img, 768, 1024), device=dev, generator=g) ** 4 * 255).to(torch.uint8)
    for _ in range(3):
        mdir_b200.clahe_u8(imgs, 4, (8, 8))
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(reps):
        mdir_b200.clahe_u8(imgs, 4, (8, 8))
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / reps
    del imgs
    out["clahe"] = {"metric": "CLAHE u8 images/s (768x1024, clip 4, 8x8 tiles)", "value": n_img / (ms * 1e-3), "unit": "images/s",
                    "batch": n_img, "ms_per_batch": ms, "algorithmic_bytes_per_image": 2 * 768 * 1024,
                    "hbm_frac_of_measured": n_img * 2 * 768 * 1024 / 1e9 / (ms * 1e-3) / peak}
    # the whole ImageClahe transform (RGB -> Lab -> CLAHE(L) -> RGB) on 32 images of 768 x 1024 x 3 float32,
    # against the reference arithmetic (cv2 float Lab conversions + cv2 CLAHE, as ImageClahe.apply) on the host
    rgbs = torch.rand((32, 768, 1024, 3), device=dev, generator=g) ** 3
    lst = list(rgbs)
    for _ in range(2):
        mdir_b200.image_clahe(lst, 4, (8, 8))
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(5):
        mdir_b200.image_clahe(lst, 4, (8, 8))
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / 5
    cpu_ms = None
    try:
        import cv2
        import numpy as np
        host = rgbs[0].cpu().numpy()
        t0 = time.perf_counter()
        for _ in range(3):
            spc = (cv2.cvtColor(host, cv2.COLOR_RGB2LAB) + np.array([0, 128, 128], np.float32)) / np.array([100.0, 255.0, 255.0], np.float32)
            spc[:, :, 0] = cv2.createCLAHE(clipLimit=4, tileGridSize=(8, 8)).apply((spc[:, :, 0] * 255).astype(np.uint8)).astype(np.float32) / 255.0
            cv2.cvtColor(spc * np.array([100.0, 255.0, 255.0], np.float32) - np.array([0, 128, 128], np.float32), cv2.COLOR_LAB2RGB)
        cpu_ms = (time.perf_counter() - t0) / 3 * 1e3
    except Exception:  # noqa: BLE001
        pass
    out["image_clahe"] = {"metric": "ImageClahe.apply (RGB->Lab->CLAHE->RGB) images/s, 768x1024x3 float32", "value": 32 / (ms * 1e-3), "unit": "images/s",
                          "ms_per_image": ms / 32, "algorithmic_bytes_per_image": 24 * 768 * 1024,
                          "hbm_frac_of_measured": 32 * 24 * 768 * 1024 / 1e9 / (ms * 1e-3) / peak,
                          "cpu_reference_ms_per_image": cpu_ms, "cpu_threads": "cv2 default"}
    del rgbs, lst
    # full (N_db, N_q) ranks: C1 shape (70 q x 4,993 x 2048, fp32-faithful scores) and a C3-shaped slice
    # (1,024 of the 10,000 queries x 100,000 x 512, bf16 scores); device-resident in and out
    from mdir_b200.search import Index
    for tag, n_db, D, nq, prec in (("ranks_c1", 4993, 2048, 70, "fp32"), ("ranks_c3_slice", 100000, 512, 1024, "bf16")):
        db = torch.randn((n_db, D), device=dev, generator=g)
        db = db / db.norm(dim=1, keepdim=True)
        q = torch.randn((nq, D), device=dev, generator=g)
        q = q / q.norm(dim=1, keepdim=True)
        idx = Index(db, device=dev, keep_fp32=(prec != "bf16"))
        for _ in range(2):
            r = idx.ranks(q, precision=prec)
        torch.cuda.synchronize()
        ev[0].record()
        for _ in range(5):
            r = idx.ranks(q, precision=prec)
        ev[1].record()
        torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1]) / 5
        pairs = n_db * nq
        out[tag] = {"metric": "full per-query ranks (scores + segmented radix sort + int64 (N_db,N_q) write)", "shape": "%d q x %d db x %d-D, %s scores" % (nq, n_db, D, prec),
                    "ms": ms, "pairs_per_s": pairs / (ms * 1e-3), "hbm_floor_frac": pairs * 12 / 1e9 / (ms * 1e-3) / peak,
                    "note": "floor = 12 B/pair (4 B score + 8 B int64 rank) at the measured HBM peak"}
        del idx, db, r
    out["c3_full"] = c3_full_measurement(torch, mdir_b200, dev, g)
    out["similarity_gemm"] = gemm_measurement(torch, dev, g)
    # SURVEY.md 8d CPU baselines beside `head` and `clahe`: the reference's torch-CPU head and OpenCV CLAHE on this host,
    # as shipped (3 torch threads / 1 cv2 thread) and on all cores
    try:
        from oracle import cpu_baselines
        cb = cpu_baselines.head_and_clahe_baselines()
        out["head"]["cpu_baseline"] = {k[5:]: v for k, v in cb.items() if k.startswith("head_")}
        out["clahe"]["cpu_baseline"] = {k[6:]: v for k, v in cb.items() if k.startswith("clahe_")}
        out["head"]["cpu_baseline"]["cores"] = out["clahe"]["cpu_baseline"]["cores"] = cb["cores"]
    except Exception as exc:  # noqa: BLE001
        out["cpu_baselines_error"] = repr(exc)
    out.update(training_side_measurements(torch, mdir_b200, dev, g, ev))
    return out


def gemm_measurement(torch, dev, g):
    """north_star: "similarity GEMM at >= 60 % of bf16 tensor peak".  The dense bf16 contraction alone
    (mdir_sim_scan_dense_bf16: tcgen05 / TMEM / TMA, (256-row tile, 128-query block) work items in one launch), as TFLOP/s
    against the measured sustained cuBLAS bf16 figure: the C3 shape (512-D: output-write-bound, 4 B out per 1,024 FLOP)
    and the tensor-bound 2048-D shape of the R1M / DBA descriptors."""
    from mdir_b200.search import Index
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    tf_sus, tf_burst = 1397.3, 1657.2
    if os.path.exists(path):
        with open(path) as fh:
            pk = json.load(fh)
            tf_sus, tf_burst = float(pk.get("bf16_tflops_sustained", tf_sus)), float(pk.get("bf16_tflops", tf_burst))
    res = {"metric": "dense bf16 similarity GEMM, fp32 scores written query-major (device-resident operands)", "unit": "TFLOP/s",
           "peak_sustained": tf_sus, "peak_burst": tf_burst, "shapes": []}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for n_db, D, nq in ((100000, 512, 1024), (100000, 2048, 4096)):
        db = torch.randn((n_db, D), device=dev, generator=g)
        db = db / db.norm(dim=1, keepdim=True)
        q = torch.randn((nq, D), device=dev, generator=g)
        q = q / q.norm(dim=1, keepdim=True)
        idx = Index(db, device=dev, keep_fp32=False)
        sc = torch.empty((nq, n_db), dtype=torch.float32, device=dev)
        for _ in range(3):
            idx.scores(q, out=sc, precision="bf16")
        torch.cuda.synchronize()
        ev[0].record()
        for _ in range(10):
            idx.scores(q, out=sc, precision="bf16")
        ev[1].record()
        torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1]) / 10
        tf = 2.0 * nq * n_db * D / (ms * 1e-3) / 1e12
        res["shapes"].append({"shape": "%d q x %d db x %d-D" % (nq, n_db, D), "ms": ms, "tflops": tf, "frac_of_sustained": tf / tf_sus,
                              "frac_of_burst": tf / tf_burst, "output_TB_per_s": nq * n_db * 4 / (ms * 1e-3) / 1e12})
        del idx, db, q, sc
    res["value"] = res["shapes"][-1]["tflops"]
    res["frac_of_sustained"] = res["shapes"][-1]["frac_of_sustained"]
    res["note"] = "ms includes the fp32 -> bf16 pack of the queries; ncu tensor-pipe evidence: profiles/r02_ncu_full_dense_gemm.json"
    return res


def c3_full_measurement(torch, mdir_b200, dev, g):
    """BASELINE.json config C3 at full size: 10,000 queries x 100,000 database rows x 512-D -> the (N_db, N_q) int64
    ranks array (8 GB) and mAP from it, everything on the device; the reference's np.dot + np.argsort timed on a
    64-query sample of the same matrices for scale."""
    import numpy as np
    from mdir_b200.search import Index
    from mdir_b200.evaluate import compute_map
    n_db, D, nq = 100000, 512, 10000
    db = torch.randn((n_db, D), device=dev, generator=g)
    db = db / db.norm(dim=1, keepdim=True)
    src = torch.randperm(n_db, device=dev, generator=g)[:nq]
    q = db[src] + 0.7 * torch.randn((nq, D), device=dev, generator=g) / D ** 0.5
    q = q / q.norm(dim=1, keepdim=True)
    src_h = src.cpu().numpy()
    rs = np.random.RandomState(11)
    gnd = [{"ok": np.array([int(src_h[i])] + rs.randint(0, n_db, 3).tolist()), "junk": rs.randint(0, n_db, 2)} for i in range(nq)]
    idx = Index(db, device=dev, keep_fp32=False)
    ranks = idx.ranks(q, precision="bf16")               # first call: cudaMalloc of the 8 GB result + 5 GB of workspace
    del ranks
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    ranks = idx.ranks(q, precision="bf16")
    ev[1].record()
    torch.cuda.synchronize()
    ms_ranks = ev[0].elapsed_time(ev[1])
    t0 = time.perf_counter()
    mp, aps, _, _ = compute_map(ranks, gnd, device=dev)
    torch.cuda.synchronize()
    ms_map = (time.perf_counter() - t0) * 1e3
    first_ok = bool((ranks[0] == src).float().mean().item() > 0.99)
    dbh, qh = db.cpu().numpy(), q[:64].cpu().numpy()
    t0 = time.perf_counter()
    np.argsort(-np.dot(dbh, qh.T), axis=0)
    cpu_ms = (time.perf_counter() - t0) * 1e3 * (nq / 64)
    del ranks, idx, db, q
    return {"metric": "C3 full size: scores + full ranks (N_db, N_q) int64 + mAP on the device", "shape": "%d q x %d db x %d-D, bf16 scores" % (nq, n_db, D),
            "ranks_ms": ms_ranks, "map_ms_incl_host_flatten": ms_map, "pairs_per_s": n_db * nq / (ms_ranks * 1e-3), "mAP": mp,
            "planted_neighbour_ranked_first": first_ok, "cpu_port_ms_dot_argsort": cpu_ms, "cpu_sample": "64 of %d queries, time scaled" % nq}


def training_side_measurements(torch, mdir_b200, dev, g, ev):
    """Row f4: hard-negative mining at the reference's default epoch shape (2000 queries x 20000 pool images,
    2048-D, 5 negatives; traindataset.py:54) and whitening learning (2048-D, 20000 images, 10000 pairs)."""
    import numpy as np
    from oracle import oracle
    out = {}
    D, n_q, n_pool, nnum = 2048, 2000, 20000, 5
    pool = torch.randn((D, n_pool), device=dev, generator=g)
    pool = pool / pool.norm(dim=0, keepdim=True)
    qv = pool[:, :n_q] + 0.05 * torch.randn((D, n_q), device=dev, generator=g)
    qv = qv / qv.norm(dim=0, keepdim=True)
    rs = np.random.RandomState(3)
    pc = rs.randint(0, 700, n_pool).astype(np.int32)
    qc = pc[:n_q].copy()
    for _ in range(2):
        mdir_b200.mine_hard_negatives(qv, pool, qc, pc, nnum, device=dev)
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(3):
        mdir_b200.mine_hard_negatives(qv, pool, qc, pc, nnum, device=dev)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / 3
    sub = 100                                              # CPU: the reference's mm + sort + walk on 100 of the 2000 queries
    ph, qh = pool.cpu().numpy(), qv[:, :sub].cpu().numpy()
    t0 = time.perf_counter()
    oracle.mine_negatives(qh, ph, qc[:sub], pc, nnum)
    cpu_ms = (time.perf_counter() - t0) * 1e3 * (n_q / sub)
    out["mining"] = {"metric": "hard-negative mining (scores + full ranks + cluster walk + distances)", "shape": "%d q x %d pool x %d-D, %d negatives" % (n_q, n_pool, D, nnum),
                     "ms": ms, "queries_per_s": n_q / (ms * 1e-3), "cpu_port_ms": cpu_ms, "cpu_sample": "%d of %d queries, time scaled" % (sub, n_q)}
    del pool, qv
    N, n_pairs = 20000, 10000
    X = torch.randn((D, N), device=dev, generator=g, dtype=torch.float32)
    X = X / X.norm(dim=0, keepdim=True)
    qi, pi = rs.randint(0, N, n_pairs), rs.randint(0, N, n_pairs)
    mdir_b200.whitenlearn(X, qi, pi, device=dev)
    torch.cuda.synchronize()
    ev[0].record()
    mdir_b200.whitenlearn(X, qi, pi, device=dev)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1])
    X64 = X.double()
    for _ in range(2):
        mdir_b200.gemm_f64(X64, X64, False)
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(3):
        mdir_b200.gemm_f64(X64, X64, False)
    ev[1].record()
    torch.cuda.synchronize()
    gms = ev[0].elapsed_time(ev[1]) / 3
    Xh = X[:512, :5000].cpu().numpy()                      # CPU: the numpy algorithm on a 512-D x 5000 slice (O(D^2 N + D^3))
    t0 = time.perf_counter()
    oracle.whitenlearn(Xh, qi[:2500] % 5000, pi[:2500] % 5000)
    cpu_ms = (time.perf_counter() - t0) * 1e3
    out["whitenlearn"] = {"metric": "whitenlearn (fp64): pair covariance, Cholesky, data covariance, eigendecomposition", "shape": "%d-D x %d images, %d pairs" % (D, N, n_pairs),
                          "ms": ms, "gemm_f64_ms_2048x2048x20000": gms, "gemm_f64_tflops": 2.0 * D * D * N / (gms * 1e-3) / 1e12,
                          "cpu_port_ms_512d_x_5000": cpu_ms,
                          "note": "O(D^2 N) contractions in mdir_gemm_f64 (SIMT DFMA); D x D factorisations are cuSOLVER via torch.linalg"}
    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
