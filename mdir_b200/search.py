"""Query x database similarity, top-k and full ranks.

Replaces, for mdir's evaluation (mdir/components/optim/score/cirscore.py:65-70):

    scores = np.dot(vecs.T, qvecs)          # (N_db, N_q)
    ranks  = np.argsort(-scores, axis=0)    # (N_db, N_q) int64

* ``rank(vecs, qvecs)``      -- the drop-in: host (D,N) matrices in, (N_db,N_q) int64 ranks out.
* ``Index``                  -- a database resident in HBM as row-major bf16 (+ optional fp32
                                master for exact re-scoring); ``search`` = tcgen05 scan with the
                                top-k selection fused into the epilogue, ``scores`` / ``ranks``
                                = the dense path.
* ``ShardedIndex``           -- rows sharded contiguously over the ranks of a torch.distributed
                                group; local top-k + one all-gather of N_q*k keys + merge.
* ``ranks_from_scores`` / ``topk_from_scores`` -- the sort/selection kernels fed an existing
                                (N_db, N_q) score matrix (bit-exact vs the stable argsort).
"""
import numpy as np
import torch

from . import _lib

TILE = 256            # MDIR_SCAN_TILE_ROWS
MAX_Q = 128           # queries per scan pass on the serving path (double / triple buffered TMEM accumulators)
DENSE_LAUNCH_Q = 1 << 20   # queries per mdir_sim_scan_dense_bf16 launch ((tile, query block) work items are counted in 30 bits)
MAX_Q_WIDE = 256      # rows of the default candidate buffers
SINGLE_GPU_SCAN_CTAS = 140   # split serving graphs on one GPU: SMs the scan keeps; the other 8 run finalize of the previous ticket
WIDE_Q = 1024         # queries per WIDE launch (search(block_q=1024): DBA, all-pairs): 8 blocks of 128 per database tile
N_SEGS = 149          # MDIR_CAND_SEGS: segment 0 = select kernel, 1 + c = scan CTA c
CAP_S = 8192          # capacity of segment 0 (the >= kth sample rows that pass, incl. ties)
CAP_L = 96            # capacity of each scan CTA's private segment
CAND_ROW = CAP_S + 148 * CAP_L
STAGE_CAP = 16384     # keys mdir_topk_finalize can stage in shared memory
MAX_SAMPLE_TILES = 512
FUSED_CAP_L = CAND_ROW // 148   # one-launch route: no select segment, so each CTA segment gets the whole row's share
TARGET_CAND = 4500    # candidates per query the sampling plan aims for (kth * n_tiles / n_sample), ~30 per CTA segment


STATUS_OVERFLOW, STATUS_UNCERTIFIED, STATUS_PEER_TIMEOUT = 1, 2, 4     # MDIR_STATUS_* (+ the exchange's own bit)
MAX_KTH = 4096        # deepest selection the finalize kernel stages
# int8 first pass (Index._i8_route): taken only when every row's int8 residual is small against the row,
# max_r ||x_r - s_r x8_r|| / ||x_r|| below this.  Unit randn rows at D = 2048 measure 0.013, where the certified bound
# (~0.013 on unit rows) keeps t - eps above the fused scan's in-kernel threshold for typical queries; a heavy-tailed
# database (a few dimensions x20) measures several times more and stays on the bf16 first pass.
I8_MAX_REL_RESIDUAL = 0.02
# ... and only on shards of at least this many rows.  Both sides of the trade shrink with the shard, but not alike.
# The scan saves n * D bytes.  The finalize re-scores ~5x as many rows in fp32, and that cost falls more slowly.  The
# certified reach t - eps also narrows: t, the k-th best score, sits lower in a smaller shard's tail, while the fused
# scan's threshold (the kth best of one sampled tile per CTA) sits higher, because the sample is a larger share.
# Measured at D = 2048, 70 queries, top-100 on a B200 (tools/time_i8_shard.py, profiles/r03_i8_shard.log):
#   125 k rows: int8 uncertified on every query;  250 k rows: 54 / 560 queries uncertified;
#   500 k / 750 k rows: certified, but 0.424 / 0.525 ms per step against bf16's 0.363 / 0.515;
#   1 M rows: 0.652 against 0.666.
I8_MIN_ROWS = 900000


def default_shortlist(k):
    """Initial bf16 shortlist for an exact fp32 top-k: 1.25 k rounded up to a multiple of 64 (whole rounds of the
    2 x 32 re-scoring warps).  It only has to be a good first guess: the finalize kernel extends it with every
    candidate whose bf16 score is within the certified error bound of the k-th fp32 score, and flags the query
    when even the candidate list is not provably deep enough (mdir_topk_finalize_rescore)."""
    return -(-(-(-5 * int(k) // 4)) // 64) * 64


def balanced_grid(n_work, max_ctas):
    """common.cuh:balanced_grid -- the smallest persistent grid that needs as many rounds as max_ctas CTAs would."""
    if n_work <= 0 or max_ctas <= 0:
        return 1
    if n_work <= max_ctas:
        return int(n_work)
    rounds = -(-n_work // max_ctas)
    return int(-(-n_work // rounds))


def _as_dev_f32(x, device):
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    if x.dtype != torch.float32:
        x = x.float()
    if x.device != device:
        x = x.pin_memory().to(device, non_blocking=True) if x.device.type == "cpu" else x.to(device)
    return x.contiguous()


def pack_bf16(x, dxn=False):
    """x fp32 cuda: (n, D) rows, or with dxn=True the reference's (D, n) -> (n, D) bf16 rows."""
    _lib.require_cuda(x, "descriptors")
    x = x.contiguous()
    if dxn:
        D, n = x.shape
    else:
        n, D = x.shape
    if D % 8:
        raise _lib.MdirError("descriptor dimension must be a multiple of 8 (got %d)" % D)
    out = torch.empty((n, D), dtype=torch.bfloat16, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().mdir_pack_bf16(_lib.ptr(x), n, D, 1 if dxn else 0, _lib.ptr(out), _lib.stream()), "mdir_pack_bf16")
    return out


class Index:
    """A (shard of a) descriptor database on one GPU."""

    fused = True      # allow the one-launch threshold + filter route (False: always sample -> select -> filter)
    certify = True    # precision="fp32": prove the shortlist complete (status bit 2 + widening when it cannot be)
    _sms = None

    def __init__(self, vecs, dxn=False, device="cuda", keep_fp32=True, idx_base=0):
        """vecs: (n, D) fp32 rows (torch/numpy, host or device), or (D, n) with dxn=True
        (the layout extract_vectors returns, cirtorch/networks/imageretrievalnet.py:291)."""
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.MdirError("Index needs a CUDA device (no CPU path)")
        v = _as_dev_f32(vecs, self.device)
        self.db16 = pack_bf16(v, dxn=dxn)
        self.n, self.D = self.db16.shape
        self.idx_base = int(idx_base)
        self.db32 = None
        if keep_fp32:
            self.db32 = v.t().contiguous() if dxn else v
        self._ws = {}
        self._stats = None
        self.db8 = self.row_scale = None
        self.route = None
        self.cert = {"queries": 0, "flagged": 0, "widened_blocks": 0, "uncertified": 0, "int8_blocks": 0, "int8_redone": 0}

    @classmethod
    def from_packed(cls, db16, db32=None, idx_base=0):
        self = cls.__new__(cls)
        self.device = db16.device
        self.db16 = db16
        self.n, self.D = db16.shape
        self.db32 = db32
        self.idx_base = int(idx_base)
        self._ws = {}
        self._stats = None
        self.db8 = self.row_scale = None
        self.route = None
        self.cert = {"queries": 0, "flagged": 0, "widened_blocks": 0, "uncertified": 0, "int8_blocks": 0, "int8_redone": 0}
        return self

    def stats(self):
        """Device float32[4] = {max_r ||bf16(x_r) - x_r||^2, max_r ||x_r||^2, max_r ||x_r - s_r x8_r||^2,
        max_r ||x_r - s_r x8_r||^2 / ||x_r||^2}: the database half of the shortlist certificate's error bound (one pass
        over the shard, cached).  When D % 128 == 0 and the shard has at least I8_MIN_ROWS rows the same pass builds the
        int8 plane of the first pass (db8, row_scale: mdir_pack_stats_i8); it is kept only when the residuals qualify
        for that route (I8_MAX_REL_RESIDUAL), which is read back to the host here, once per index.  Otherwise the last
        two entries are 0."""
        if self._stats is None:
            if self.db32 is None:
                raise _lib.MdirError("the shortlist certificate needs the fp32 master copy (keep_fp32=True)")
            st = torch.zeros((4,), dtype=torch.float32, device=self.device)
            lib = _lib.lib()
            with torch.cuda.device(self.device):
                if self.D % 128 == 0 and self.n >= I8_MIN_ROWS:
                    db8 = torch.empty((self.n, self.D), dtype=torch.int8, device=self.device)
                    rs = torch.empty((self.n,), dtype=torch.float32, device=self.device)
                    _lib.check(lib.mdir_pack_stats_i8(_lib.ptr(self.db32), _lib.ptr(self.db16), self.n, self.D, _lib.ptr(st), _lib.ptr(db8),
                                                      _lib.ptr(rs), _lib.stream()), "mdir_pack_stats_i8")
                    if float(st[3].item()) < I8_MAX_REL_RESIDUAL ** 2:
                        self.db8, self.row_scale = db8, rs
                else:
                    _lib.check(lib.mdir_pack_stats(_lib.ptr(self.db32), _lib.ptr(self.db16), self.n, self.D, _lib.ptr(st), _lib.stream()),
                               "mdir_pack_stats")
            self._stats = st
        return self._stats

    # ------------------------------------------------------------------ helpers
    def _buf(self, name, shape, dtype):
        key = (getattr(self, "_ws_tag", None), name, tuple(shape), dtype)      # _ws_tag: a private workspace set (GraphedSearch(split=True))
        b = self._ws.get(key)
        if b is None:
            b = torch.empty(shape, dtype=dtype, device=self.device)
            self._ws[key] = b
        return b

    def _plan(self, kth):
        """Sampling plan for the threshold pass: (n_sample, stride) or None for the dense route.
        The threshold is the kth best of n_sample*256 sampled rows, so about kth * n_tiles / n_sample
        rows survive the filter pass; n_sample is sized to keep that near TARGET_CAND."""
        n_tiles = (self.n + TILE - 1) // TILE
        if n_tiles < 64:
            return None
        want = -(-kth * n_tiles // TARGET_CAND)                     # ceil
        if want > 148:                                              # whole waves of the 148 persistent CTAs
            want = -(-want // 148) * 148
        n_sample = max(32, min(MAX_SAMPLE_TILES, n_tiles // 4, want))
        stride = n_tiles // n_sample
        if n_sample * TILE < 2 * kth or stride < 2:
            return None
        return n_sample, stride

    def _fused_ok(self, kth, nq=1):
        """One-launch route (mdir_sim_scan_fused_bf16): each of the g persistent CTAs samples one tile, so the
        threshold is about the kth best of g*256 rows and ~1.25 * kth * n_tiles / g rows survive, spread over g
        segments.  Taken when that keeps the segments at most half full; larger k or databases use the
        three-launch route, whose sample grows with the database."""
        if not self.fused or nq > MAX_Q:
            return False
        n_tiles = (self.n + TILE - 1) // TILE
        if self._sms is None:
            self._sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        g = balanced_grid(n_tiles, min(148, self._sms, n_tiles // 2))
        if n_tiles < 64 or g * 16 < 2 * kth:
            return False
        return 1.25 * kth * n_tiles / (g * g) <= FUSED_CAP_L / 2

    def _i8_route(self, kth, nq):
        """The int8 first pass (mdir_pack_q_i8 -> mdir_sim_scan_fused_i8 -> mdir_topk_finalize_rescore_eps): half the
        database bytes of the bf16 scan.  Taken for a certified fp32 search on the one-launch route when the shard
        has an int8 plane (D % 128 == 0, at least I8_MIN_ROWS rows and small int8 residuals, see stats()).  Its bound is wider than bf16's, so it
        never widens: a flagged block is redone through the bf16 route (Index._run_block)."""
        if not (self.certify and self.db32 is not None and self.D % 128 == 0 and self._fused_ok(kth, nq)):
            return False
        self.stats()
        return self.db8 is not None

    def _fused_ws(self):
        ws = self._ws.get("fused_ws")
        if ws is None:                       # zeroed once; the kernel re-arms its arrival counters itself
            ws = torch.zeros((_lib.lib().mdir_sim_scan_fused_workspace_bytes(MAX_Q) // 4,), dtype=torch.int32, device=self.device)
            self._ws["fused_ws"] = ws
        return ws

    def _topk_block_i8(self, q32, kth, k_out, out_scores, out_idx, out_keys, ovf):
        """The certified fp32 top-k_out of one block of <= 128 queries through the int8 first pass: three launches."""
        lib = _lib.lib()
        nq = q32.shape[0]
        n_pad = -(-nq // 16) * 16
        stats = self.stats()
        q8 = self._buf("q8", (2 * n_pad, self.D), torch.int8)
        qsc = self._buf("q8_scale", (nq, 2), torch.float32)
        qeps = self._buf("q8_eps", (nq,), torch.float32)
        _lib.check(lib.mdir_pack_q_i8(_lib.ptr(q32), nq, self.D, _lib.ptr(stats), _lib.ptr(q8), _lib.ptr(qsc), _lib.ptr(qeps), _lib.stream()),
                   "mdir_pack_q_i8")
        tau, cand, cnt = self._cand_bufs(nq)
        ws = self._fused_ws()
        prof = getattr(self, "prof", None)
        if prof is not None:
            prof.begin()
        _lib.check(lib.mdir_sim_scan_fused_i8(_lib.ptr(self.db8), _lib.ptr(self.row_scale), self.n, _lib.ptr(q8), _lib.ptr(qsc), nq, self.D, kth,
                                              _lib.ptr(tau), self.idx_base, _lib.ptr(cand), _lib.ptr(cnt), 0, FUSED_CAP_L, _lib.ptr(ws),
                                              _lib.stream()), "mdir_sim_scan_fused_i8")
        if prof is not None:
            prof.end(self.n * self.D + 4 * self.n)       # int8 rows + their fp32 scales
        self._finalize(cand, cnt, nq, kth, out_scores, out_idx, out_keys, tau, ovf, (q32, k_out), caps=(0, FUSED_CAP_L), q_eps=qeps)

    def _scan(self, q16, mode, stride, n_sample, dense, dense_ld, tau, cand, cnt):
        # more than 128 queries: one WIDE launch, work items = (tile, 128-query block) -- one kernel ramp, and a database
        # tile comes from HBM once for all the blocks (the tensor-bound regime: DBA, all-pairs)
        fn = _lib.lib().mdir_sim_scan_wide_bf16 if q16.shape[0] > MAX_Q else _lib.lib().mdir_sim_scan_bf16
        _lib.check(fn(_lib.ptr(self.db16), self.n, _lib.ptr(q16), q16.shape[0], self.D, mode, stride,
                      n_sample, _lib.ptr(dense), dense_ld, _lib.ptr(tau), self.idx_base, _lib.ptr(cand),
                      _lib.ptr(cnt), CAP_S, CAP_L, _lib.stream()), "mdir_sim_scan_bf16")

    def _cand_bufs(self, nq=MAX_Q_WIDE):
        rows = MAX_Q_WIDE if nq <= MAX_Q_WIDE else WIDE_Q
        return (self._buf("tau", (rows,), torch.int64), self._buf("cand", (rows, CAND_ROW), torch.int64),
                self._buf("segcnt", (rows, N_SEGS), torch.int32))

    def _finalize(self, cand, cnt, nq, kth, out_scores, out_idx, out_keys, tau, ovf, rescore=None, caps=(CAP_S, CAP_L), q_eps=None):
        """rescore = (q32_block, k_out): fused exact fp32 re-scoring of the kth-long bf16 shortlist.
        q_eps: per-query bounds of the int8 first pass (certified, instead of the bf16 bound)."""
        CAP_S, CAP_L = caps
        CAND_ROW = CAP_S + 148 * CAP_L            # the row stride the scan kernels derive from the two capacities
        if rescore is None:
            _lib.check(_lib.lib().mdir_topk_finalize(_lib.ptr(cand), CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, CAP_L, nq, kth,
                                                     _lib.ptr(out_scores), _lib.ptr(out_idx), _lib.ptr(out_keys), _lib.ptr(tau),
                                                     _lib.ptr(ovf), _lib.stream()), "mdir_topk_finalize")
        elif q_eps is not None:
            q32, k_out = rescore
            _lib.check(_lib.lib().mdir_topk_finalize_rescore_eps(_lib.ptr(cand), CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, CAP_L, nq, kth, k_out,
                                                                 _lib.ptr(self.db32), self.n, self.idx_base, _lib.ptr(q32), self.D,
                                                                 _lib.ptr(self.stats()), _lib.ptr(q_eps), _lib.ptr(out_scores), _lib.ptr(out_idx),
                                                                 _lib.ptr(out_keys), _lib.ptr(tau), _lib.ptr(ovf), _lib.stream()),
                       "mdir_topk_finalize_rescore_eps")
        else:
            q32, k_out = rescore
            stats = self.stats() if self.certify else None
            _lib.check(_lib.lib().mdir_topk_finalize_rescore(_lib.ptr(cand), CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, CAP_L, nq, kth, k_out,
                                                             _lib.ptr(self.db32), self.n, self.idx_base, _lib.ptr(q32), self.D,
                                                             _lib.ptr(stats), _lib.ptr(out_scores), _lib.ptr(out_idx), _lib.ptr(out_keys),
                                                             _lib.ptr(tau), _lib.ptr(ovf), _lib.stream()), "mdir_topk_finalize_rescore")

    def _dense_block(self, q16, kth, out_scores, out_idx, out_keys, ovf, rescore=None):
        """All scores of the block -> exact kth-key select -> sort.  The route for small databases
        and the guaranteed-terminating recovery when a candidate segment overflowed (the select
        emits exactly kth keys, so nothing can overflow here)."""
        lib = _lib.lib()
        nq = q16.shape[0]
        tau, cand, cnt = self._cand_bufs(nq)     # the select kernel (re)initialises every segment counter
        dense = self._buf("dense", (MAX_Q if nq <= MAX_Q else (MAX_Q_WIDE if nq <= MAX_Q_WIDE else WIDE_Q), max(self.n, 1)), torch.float32)
        self._scan(q16, 0, 0, 0, dense, self.n, None, None, None)
        _lib.check(lib.mdir_select_kth(_lib.ptr(dense), self.n, self.n, nq, kth, 0, self.idx_base, _lib.ptr(tau),
                                       _lib.ptr(cand), CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, 0, _lib.stream()), "mdir_select_kth")
        self._finalize(cand, cnt, nq, kth, out_scores, out_idx, out_keys, tau, ovf, rescore)

    def _topk_block(self, q16, kth, out_scores, out_idx, out_keys, ovf, rescore=None):
        """Exact top-kth of one block of <= 128 queries by bf16-input/fp32-accumulate scores."""
        lib = _lib.lib()
        nq = q16.shape[0]
        plan = self._plan(kth)
        if plan is None:
            return self._dense_block(q16, kth, out_scores, out_idx, out_keys, ovf, rescore)
        tau, cand, cnt = self._cand_bufs(nq)     # the select / fused kernel (re)initialises every segment counter
        prof = getattr(self, "prof", None)       # bench.py: CUDA events around the dominant kernel, on its own stream
        if self._fused_ok(kth, nq):
            ws = self._fused_ws()
            if prof is not None:
                prof.begin()
            _lib.check(lib.mdir_sim_scan_fused_bf16(_lib.ptr(self.db16), self.n, _lib.ptr(q16), nq, self.D, kth, _lib.ptr(tau),
                                                    self.idx_base, _lib.ptr(cand), _lib.ptr(cnt), 0, FUSED_CAP_L, _lib.ptr(ws),
                                                    _lib.stream()), "mdir_sim_scan_fused_bf16")
            if prof is not None:
                prof.end(self.n * self.D * 2)
            return self._finalize(cand, cnt, nq, kth, out_scores, out_idx, out_keys, tau, ovf, rescore, caps=(0, FUSED_CAP_L))
        n_sample, stride = plan
        rows = n_sample * TILE
        if nq <= MAX_Q_WIDE:
            sample = self._buf("sample", (MAX_Q if nq <= MAX_Q else MAX_Q_WIDE, MAX_SAMPLE_TILES * TILE), torch.float32)
            ld = MAX_SAMPLE_TILES * TILE
        else:
            sample = self._buf("sample_wide", (WIDE_Q, rows), torch.float32)
            ld = rows
        self._scan(q16, 1, stride, n_sample, sample, ld, None, None, None)
        _lib.check(lib.mdir_select_kth(_lib.ptr(sample), ld, rows, nq, kth, stride, self.idx_base, _lib.ptr(tau),
                                       _lib.ptr(cand), CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, 1, _lib.stream()), "mdir_select_kth")
        if prof is not None:
            prof.begin()
        self._scan(q16, 2, stride, n_sample, None, 0, tau, cand, cnt)
        if prof is not None:
            prof.end((self.n - rows) * self.D * 2)
        self._finalize(cand, cnt, nq, kth, out_scores, out_idx, out_keys, tau, ovf, rescore)

    # ------------------------------------------------------------------ public
    def search(self, q, k, precision="fp32", shortlist=None, check=True, return_keys=False, block_q=MAX_Q):
        """q: (N_q, D) fp32 (host or device).  Returns (scores (N_q,k) fp32, idx (N_q,k) int32) on
        the device, ordered by (score desc, index asc); idx = idx_base + local row, -1 padding.

        precision="bf16": exact top-k of the bf16-input / fp32-accumulate scores.
        precision="fp32": bf16 shortlist of `shortlist` (default 1.25 k rounded up to 64) per query, re-scored exactly in
                          fp32 against the fp32 master copy and extended until certified (mdir_topk_finalize_rescore).
        check=False skips the (synchronising) status check; call check_overflow() later.
        block_q: queries per scan pass, 128 (serving) up to 1,024 (tensor-bound batches -- DBA, all-pairs: one WIDE launch,
        (tile, 128-query block) work items, the database streamed from HBM once per 1,024 queries)."""
        lib = _lib.lib()
        with torch.cuda.device(self.device):
            q32 = _as_dev_f32(q, self.device)
            nq_all = q32.shape[0]
            if q32.shape[1] != self.D:
                raise _lib.MdirError("query dimension %d != database dimension %d" % (q32.shape[1], self.D))
            k = int(k)
            if nq_all == 0:
                empty = (torch.empty((0, k), dtype=torch.float32, device=self.device), torch.empty((0, k), dtype=torch.int32, device=self.device))
                return empty + (torch.empty((0, k), dtype=torch.int64, device=self.device),) if return_keys else empty
            k_eff = min(k, self.n)
            if precision == "fp32":
                if self.db32 is None:
                    raise _lib.MdirError("precision='fp32' needs keep_fp32=True")
                kth = max(k_eff, min(self.n, int(shortlist or default_shortlist(k))))
            elif precision == "bf16":
                kth = k_eff
            else:
                raise ValueError("precision must be 'fp32' or 'bf16'")
            if kth > 4096:
                raise _lib.MdirError("k/shortlist %d too large for the fused path (max 4096); use ranks()" % kth)
            q16 = None                          # bf16 queries: packed on the first block that takes a bf16 route
            out_s = torch.empty((nq_all, k), dtype=torch.float32, device=self.device)
            out_i = torch.empty((nq_all, k), dtype=torch.int32, device=self.device)
            out_k = torch.empty((nq_all, k), dtype=torch.int64, device=self.device) if return_keys else None
            self._ovf = self._buf("ovf", (max(nq_all, 1),), torch.int32)
            block_q = max(MAX_Q, min(WIDE_Q, int(block_q)))
            for q0 in range(0, nq_all, block_q):
                q1 = min(q0 + block_q, nq_all)
                nq = q1 - q0
                ovf = self._ovf[q0:q1]
                bs, bi = out_s[q0:q1], out_i[q0:q1]
                bk = out_k[q0:q1] if return_keys else None
                rescore = (q32[q0:q1], k_eff) if precision == "fp32" else None
                kk = kth if precision == "fp32" else k_eff
                qb = None                       # None: the int8 first pass (_run_block)
                if rescore is None or not self._i8_route(kk, nq):
                    if q16 is None:
                        q16 = pack_bf16(q32)
                    qb = q16[q0:q1]
                if k_eff < k:          # database smaller than k: pad the columns beyond it
                    bs.fill_(float("-inf")); bi.fill_(-1)
                    if bk is not None:
                        bk.fill_(-1)
                    tmp_s = torch.empty((nq, k_eff), dtype=torch.float32, device=self.device)
                    tmp_i = torch.empty((nq, k_eff), dtype=torch.int32, device=self.device)
                    tmp_k = torch.empty((nq, k_eff), dtype=torch.int64, device=self.device)
                    self._run_block(qb, kk, tmp_s, tmp_i, tmp_k, ovf, check, rescore=rescore)
                    bs[:, :k_eff] = tmp_s; bi[:, :k_eff] = tmp_i
                    if bk is not None:
                        bk[:, :k_eff] = tmp_k
                else:
                    self._run_block(qb, kk, bs, bi, bk, ovf, check, rescore=rescore)
            if return_keys:
                return out_s, out_i, out_k
            return out_s, out_i

    def _run_block(self, q16, kth, out_s, out_i, out_k, ovf, check, rescore=None):
        """q16 None: the int8 first pass (Index._i8_route); a block it flags (bit 0 or 1) is redone here through the
        bf16 route when check=True -- the int8 pass never widens, recovery is the bf16 route's own."""
        if q16 is None:
            self.route = "int8"
            self.cert["int8_blocks"] += 1
            self._topk_block_i8(rescore[0], kth, rescore[1], out_s, out_i, out_k, ovf)
            if not check:
                return
            st = ovf.cpu()
            if not bool(st.any()):
                self.cert["queries"] += int(st.numel())
                return
            self.cert["int8_redone"] += 1
            q16 = pack_bf16(rescore[0])
        self.route = "bf16"
        self._topk_block(q16, kth, out_s, out_i, out_k, ovf, rescore)
        if not check:
            return
        st = ovf.cpu()
        self.cert["queries"] += int(st.numel())
        if bool((st & STATUS_OVERFLOW).any()):
            # a candidate segment overflowed (adversarial row order / massive ties): exact dense route
            self._dense_block(q16, kth, out_s, out_i, out_k, ovf, rescore)
            st = ovf.cpu()
            if bool((st & STATUS_OVERFLOW).any()):
                raise _lib.MdirError("dense recovery overflowed (internal error)")
        if rescore is None:
            return
        self.cert["flagged"] += int((st & STATUS_UNCERTIFIED).ne(0).sum())
        # the shortlist certificate failed for some query: the candidate list was not provably deep enough.  Widen the
        # selection (x2 per round; deeper kth = lower threshold = more candidates) until it is, at most MAX_KTH rows.
        k_max = min(self.n, MAX_KTH)
        while bool((st & STATUS_UNCERTIFIED).any()) and kth < k_max:
            kth = min(2 * kth, k_max)
            self.cert["widened_blocks"] += 1
            self._topk_block(q16, kth, out_s, out_i, out_k, ovf, rescore)
            st = ovf.cpu()
            if bool((st & STATUS_OVERFLOW).any()):
                self._dense_block(q16, kth, out_s, out_i, out_k, ovf, rescore)
                st = ovf.cpu()
        # still flagged: more than ~MAX_KTH rows lie within the error bound of the k-th score (massive near-ties).
        # The best-effort answer stands; the flag stays raised in status() and the counter records it.
        self.cert["uncertified"] += int((st & STATUS_UNCERTIFIED).ne(0).sum())

    def check_overflow(self):
        """True if the last search(check=False) raised a status flag for some query (candidate overflow or a failed
        shortlist certificate): rerun that batch through search(check=True), which recovers / widens."""
        return bool(self._ovf.any().item())

    def status(self):
        """Per-query status words of the last search (0 = exact and, for precision='fp32', certified)."""
        return self._ovf

    def _split3(self, x, role):
        """(n, D) fp32 -> (n, 3D) fp32 [hi|hi|lo] (role 0) / [hi|lo|hi] (role 1) for the 3xTF32 scan."""
        n, D = x.shape
        out = torch.empty((n, 3 * D), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().mdir_split_tf32x3(_lib.ptr(x), n, D, role, _lib.ptr(out), _lib.stream()), "mdir_split_tf32x3")
        return out

    def scores(self, q, out=None, precision="bf16"):
        """Dense scores, QUERY-major: (N_q, N_db) fp32 on the device.
        precision "bf16": bf16 operands, fp32 accumulate (|err| <~ 1e-3 on unit vectors);
                  "tf32": fp32 operands consumed as TF32 by the tensor cores;
                  "fp32": 3xTF32 split (hi*hi + hi*lo + lo*hi) = fp32-faithful (|err| ~ 1e-6);
        tf32 / fp32 need the fp32 master copy (keep_fp32=True); fp32 caches a 3x-wide split of it."""
        lib = _lib.lib()
        with torch.cuda.device(self.device):
            q32 = _as_dev_f32(q, self.device)
            nq_all = q32.shape[0]
            if out is None:
                out = torch.empty((nq_all, self.n), dtype=torch.float32, device=self.device)
            if precision == "bf16":
                q16 = pack_bf16(q32)
                if nq_all > MAX_Q and out.stride(0) >= self.n and self.n > 0:
                    # every 128-query block in one launch (one kernel ramp, the database streamed once)
                    for q0 in range(0, nq_all, DENSE_LAUNCH_Q):
                        q1 = min(q0 + DENSE_LAUNCH_Q, nq_all)
                        _lib.check(lib.mdir_sim_scan_dense_bf16(_lib.ptr(self.db16), self.n, _lib.ptr(q16[q0:q1]), q1 - q0, self.D,
                                                                _lib.ptr(out[q0:q1]), out.stride(0), _lib.stream()), "mdir_sim_scan_dense_bf16")
                    return out
                for q0 in range(0, nq_all, MAX_Q):
                    q1 = min(q0 + MAX_Q, nq_all)
                    self._scan(q16[q0:q1], 0, 0, 0, out[q0:q1], out.stride(0), None, None, None)
                return out
            if precision not in ("tf32", "fp32"):
                raise ValueError("precision must be 'bf16', 'tf32' or 'fp32'")
            if self.db32 is None:
                raise _lib.MdirError("precision=%r needs keep_fp32=True" % precision)
            if precision == "tf32":
                dbx, qx, D = self.db32, q32, self.D
            else:
                if getattr(self, "_db_x3", None) is None:
                    self._db_x3 = self._split3(self.db32, 0)
                dbx, qx, D = self._db_x3, self._split3(q32, 1), 3 * self.D
            for q0 in range(0, nq_all, MAX_Q):
                q1 = min(q0 + MAX_Q, nq_all)
                _lib.check(lib.mdir_sim_scan_tf32(_lib.ptr(dbx), self.n, _lib.ptr(qx[q0:q1]), q1 - q0, D, 0, 0, 0, _lib.ptr(out[q0:q1]),
                                                  self.n, None, self.idx_base, None, None, 0, 0, _lib.stream()), "mdir_sim_scan_tf32")
            return out

    def ranks(self, q, max_pairs=1 << 28, precision="bf16"):
        """Full ranking: (N_db, N_q) int64 C-order on the device (== np.argsort(-scores, axis=0,
        kind='stable') of this index's scores at the given precision, see scores()).  Queries are processed in chunks of at most
        max_pairs // N_db to bound the sort workspace (~30 B per pair)."""
        lib = _lib.lib()
        with torch.cuda.device(self.device):
            q32 = _as_dev_f32(q, self.device)
            nq_all = q32.shape[0]
            out = torch.empty((self.n, nq_all), dtype=torch.int64, device=self.device)
            if nq_all == 0 or self.n == 0:
                return out
            chunk = max(1, min(nq_all, max_pairs // max(self.n, 1)))
            chunk = max(1, min(chunk, 65535))
            ws = _rank_workspace(self.n, chunk, self.device)
            sc = torch.empty((chunk, self.n), dtype=torch.float32, device=self.device)
            starts = list(range(0, nq_all, chunk))
            status = torch.zeros((len(starts),), dtype=torch.int32, device=self.device)
            for c, q0 in enumerate(starts):
                q1 = min(q0 + chunk, nq_all)
                self.scores(q32[q0:q1], out=sc[:q1 - q0], precision=precision)
                _lib.check(lib.mdir_rank_scores_hist(_lib.ptr(sc), self.n, q1 - q0, 1, _lib.ptr(out[:, q0:]), nq_all, _lib.ptr(ws),
                                                     _lib.ptr(status[c:]), _lib.stream()), "mdir_rank_scores_hist")
            RANK_STATS["fast"] += len(starts)
            # ONE read-back for the whole call, after everything is queued; a chunk the histogram sort flagged (a bucket
            # of massive ties) is redone through the sample sort, and through the segmented radix sort if that cannot
            # stage a bucket either
            for c, st in enumerate(status.cpu().tolist()):
                if not st:
                    continue
                q0 = starts[c]
                q1 = min(q0 + chunk, nq_all)
                self.scores(q32[q0:q1], out=sc[:q1 - q0], precision=precision)
                _rank_scores_slow(sc, self.n, q1 - q0, 1, out[:, q0:], nq_all, ws, st)
            return out


RANK_STATS = {"fast": 0, "sample_sort": 0, "fallback": 0}       # histogram-sort calls / re-run through the sample sort / through the radix sort


def _rank_workspace(n_db, n_q, device):
    lib = _lib.lib()
    return torch.empty(max(lib.mdir_rank_workspace_bytes(n_db, n_q), lib.mdir_rank_fast_workspace_bytes(n_db, n_q),
                           lib.mdir_rank_hist_workspace_bytes(n_db, n_q)) + 256,
                       dtype=torch.uint8, device=device)


def _rank_scores_slow(scores, n_db, n_q, query_major, out, out_ld, ws, status):
    """The fallbacks behind a non-zero status word of mdir_rank_scores_hist: bit 1 -> sample sort (splits ties by row);
    bit 0 (from the sample sort) -> segmented LSD radix sort, which always completes."""
    lib = _lib.lib()
    if status & 2:
        RANK_STATS["sample_sort"] += 1
        st = torch.empty((1,), dtype=torch.int32, device=scores.device)
        _lib.check(lib.mdir_rank_scores_fast(_lib.ptr(scores), n_db, n_q, query_major, _lib.ptr(out), out_ld, _lib.ptr(ws), _lib.ptr(st),
                                             _lib.stream()), "mdir_rank_scores_fast")
        status = int(st.item())
    if status & 1:
        RANK_STATS["fallback"] += 1
        _lib.check(lib.mdir_rank_scores(_lib.ptr(scores), n_db, n_q, query_major, _lib.ptr(out), out_ld, _lib.ptr(ws), _lib.stream()),
                   "mdir_rank_scores")


def _rank_scores(scores, n_db, n_q, query_major, out, out_ld, ws):
    """mdir_rank_scores_hist (histogram sort), then the sample sort / the segmented radix sort when it reports a bucket it
    could not stage (one status word read back per call: the price of never returning an incomplete ranking)."""
    lib = _lib.lib()
    status = torch.empty((1,), dtype=torch.int32, device=scores.device)
    _lib.check(lib.mdir_rank_scores_hist(_lib.ptr(scores), n_db, n_q, query_major, _lib.ptr(out), out_ld, _lib.ptr(ws), _lib.ptr(status),
                                         _lib.stream()), "mdir_rank_scores_hist")
    RANK_STATS["fast"] += 1
    st = int(status.item())
    if st:
        _rank_scores_slow(scores, n_db, n_q, query_major, out, out_ld, ws, st)


def ranks_from_scores(scores, device="cuda", method="auto"):
    """scores (N_db, N_q) fp32 in the reference layout (host or device) -> ranks (N_db, N_q) int64
    on the device, bit-identical to np.argsort(-scores, axis=0, kind='stable').
    method: "auto" = sample sort with the radix sort as its fallback, "radix" = the segmented LSD radix sort only."""
    lib = _lib.lib()
    dev = torch.device(device)
    s = _as_dev_f32(scores, dev)
    n_db, n_q = s.shape
    with torch.cuda.device(dev):
        out = torch.empty((n_db, n_q), dtype=torch.int64, device=dev)
        if n_db == 0 or n_q == 0:
            return out
        for q0 in range(0, n_q, 65535):
            q1 = min(n_q, q0 + 65535)
            blk = s if (q0 == 0 and q1 == n_q) else s[:, q0:q1].contiguous()
            ws = _rank_workspace(n_db, q1 - q0, dev)
            if method == "radix":
                _lib.check(lib.mdir_rank_scores(_lib.ptr(blk), n_db, q1 - q0, 0, _lib.ptr(out[:, q0:]), n_q, _lib.ptr(ws), _lib.stream()),
                           "mdir_rank_scores")
            else:
                _rank_scores(blk, n_db, q1 - q0, 0, out[:, q0:], n_q, ws)
    return out


def topk_from_scores(scores, k, device="cuda"):
    """scores (N_db, N_q) fp32 -> (idx (k, N_q) int64, val (k, N_q) fp32) on the device: the first
    k rows of ranks_from_scores without sorting the rest (radix-select the kth score, gather
    everything that ties or beats it, sort those).  Falls back to the full sort when more rows tie
    with the kth score than the candidate buffer holds."""
    lib = _lib.lib()
    dev = torch.device(device)
    s = _as_dev_f32(scores, dev)
    n_db, n_q = s.shape
    k = int(k)
    if k > min(n_db, 4096):
        r = ranks_from_scores(s, device=dev)[:k]
        return r, torch.gather(s, 0, r)
    cap = int(min(STAGE_CAP, max(4 * k, 1024)))
    with torch.cuda.device(dev):
        st = s.t().contiguous()                       # query-major for coalesced selection
        tau = torch.empty((n_q,), dtype=torch.int64, device=dev)
        cand = torch.empty((n_q, cap), dtype=torch.int64, device=dev)
        cnt = torch.zeros((n_q,), dtype=torch.int32, device=dev)
        out_s = torch.empty((n_q, k), dtype=torch.float32, device=dev)
        out_i = torch.empty((n_q, k), dtype=torch.int32, device=dev)
        _lib.check(lib.mdir_select_kth(_lib.ptr(st), n_db, n_db, n_q, k, 0, 0, _lib.ptr(tau), _lib.ptr(cand), cap, _lib.ptr(cnt), 1, cap, 0,
                                       _lib.stream()), "mdir_select_kth")
        _lib.check(lib.mdir_topk_finalize(_lib.ptr(cand), cap, _lib.ptr(cnt), 1, cap, 0, n_q, k, _lib.ptr(out_s), _lib.ptr(out_i), None,
                                          None, None, _lib.stream()), "mdir_topk_finalize")
        if int(cnt.max().item()) > cap:               # too many exact ties at the kth score
            r = ranks_from_scores(s, device=dev)[:k]
            return r, torch.gather(s, 0, r)
    return out_i.t().contiguous().long(), out_s.t().contiguous()


def rank(vecs, qvecs, device="cuda", precision="fp32"):
    """The drop-in for cirscore.py:69-70.  vecs (D, N_db), qvecs (D, N_q): fp32 numpy/torch host
    matrices as extract_vectors returns them.  -> ranks (N_db, N_q) int64 numpy, C-order.
    The default precision "fp32" (3xTF32 on the tensor cores) reproduces the reference's fp32
    scores to ~1e-6, so the ranks differ from it only inside fp32 summation noise; "bf16" is the
    fast path (ranks may swap where scores are within ~1e-3)."""
    dev = torch.device(device)
    index = Index(vecs, dxn=True, device=dev, keep_fp32=(precision != "bf16"))
    q = _as_dev_f32(qvecs, dev).t().contiguous()
    return index.ranks(q, precision=precision).cpu().numpy()


class ShardedIndex:
    """Database rows sharded contiguously over a torch.distributed group (one process per GPU):
    shard g = rows [g*ceil(N/G), ...).  search() = local fused top-k, ONE all-gather of
    N_q*k 64-bit keys per rank (NCCL over NVLink), merge by (score desc, index asc): identical to
    the single-GPU answer by construction.  There is no other collective on the data path."""

    p2p = True            # exchange + merge in one kernel over NVLink peer memory (False: ncclAllGather + merge kernel)
    P2P_MAX_Q, P2P_MAX_K = 128, 1024

    def __init__(self, local_vecs, idx_base, group=None, device="cuda", keep_fp32=True, dxn=False):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.local = Index(local_vecs, dxn=dxn, device=device, keep_fp32=keep_fp32, idx_base=idx_base)
        self.device = self.local.device
        self._p2p_setup()

    @classmethod
    def from_local(cls, local_index, group=None):
        """Wrap an already-built local shard (its idx_base = first global row it owns)."""
        import torch.distributed as dist
        self = cls.__new__(cls)
        self.dist = dist
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.local = local_index
        self.device = local_index.device
        self._p2p_setup()
        return self

    def _p2p_setup(self):
        """Mailboxes for mdir_shard_exchange_merge: one cudaMalloc'ed buffer per rank, mapped into every peer through
        cudaIpc handles exchanged with one all-gather (setup time only).  Any failure (no peer access, a backend
        without device tensors) leaves the NCCL all-gather route in place."""
        self._mb, self._mb_own, self._mb_keep = None, None, None
        dist = self.dist
        if not (self.p2p and self.world > 1 and self.world <= 16 and self.device.type == "cuda" and dist.get_backend(self.group) == "nccl"):
            return
        import ctypes as C
        lib = _lib.lib()
        rank = dist.get_rank(self.group)
        ok = 1
        own = C.c_void_p(0)
        handle = (C.c_ubyte * 64)()
        with torch.cuda.device(self.device):
            nbytes = lib.mdir_shard_mailbox_bytes(self.world, self.P2P_MAX_Q, self.P2P_MAX_K)
            if lib.mdir_p2p_alloc(nbytes, C.byref(own), handle) != 0:
                ok = 0
            mine = torch.tensor(list(bytes(handle)) + [ok], dtype=torch.uint8, device=self.device)
            allh = torch.empty((self.world, 65), dtype=torch.uint8, device=self.device)
            dist.all_gather_into_tensor(allh.view(-1), mine, group=self.group)
            allh = allh.cpu().numpy()
            ptrs = (C.c_void_p * self.world)()
            good = bool(allh[:, 64].all())
            if good:
                for r in range(self.world):
                    if r == rank:
                        ptrs[r] = own.value
                        continue
                    peer = C.c_void_p(0)
                    hb = (C.c_ubyte * 64)(*[int(x) for x in allh[r, :64]])
                    if lib.mdir_p2p_open(hb, C.byref(peer)) != 0:
                        good = False
                        break
                    ptrs[r] = peer.value
            flag = torch.tensor([1 if good else 0], dtype=torch.int32, device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)          # all or nobody
            if int(flag.item()) == 1:
                self._mb, self._mb_own, self._rank = ptrs, own, rank
            torch.cuda.synchronize(self.device)

    def close(self):
        """Unmap the peers' mailboxes and free the own one (every rank, after the last search; optional at exit)."""
        if self._mb is None:
            return
        lib = _lib.lib()
        torch.cuda.synchronize(self.device)
        self.dist.barrier(group=self.group)                # nobody is still pushing into a mailbox about to disappear
        for r in range(self.world):
            if r != self._rank:
                lib.mdir_p2p_close(self._mb[r])
        lib.mdir_p2p_free(self._mb_own)
        self._mb, self._mb_own = None, None

    def exchange_status(self):
        """0 = healthy; 1 = a peer did not arrive within the bounded wait of some step (results of that step are padding)."""
        if self._mb is None:
            return 0
        import ctypes as C
        st = C.c_int(0)
        _lib.check(_lib.lib().mdir_shard_status(self._mb_own, C.byref(st)), "mdir_shard_status")
        return int(st.value)

    @staticmethod
    def shard_bounds(n_total, world, rank):
        per = (n_total + world - 1) // world
        lo = min(rank * per, n_total)
        return lo, min(lo + per, n_total)

    def search(self, q, k, precision="fp32", shortlist=None, check=True, exchange="sync"):
        """exchange="sync": the merged global top-k of THIS call.  exchange="deferred" (peer-memory route only, at most
        128 queries): pushes this call's keys and returns the merged result of the PREVIOUS deferred call with the same
        (n_q, k) -- its keys arrived a whole step ago, so neither the exchange latency nor the skew between ranks is
        ever waited for; drain() returns the last one.
        status() afterwards = OR over all ranks of the per-query status words of the merged step (identical on every
        rank): with check=False a rank whose candidate lists overflowed, or whose shortlist certificate failed, marks
        the query for EVERY rank instead of being merged silently."""
        s, i, keys = self.local.search(q, k, precision=precision, shortlist=shortlist, check=check, return_keys=True)
        nq_all = keys.shape[0]
        local_status = self.local._ovf[:nq_all]
        if self.world == 1:
            self._status = local_status
            return s, i
        if exchange not in ("sync", "deferred"):
            raise ValueError("exchange must be 'sync' or 'deferred'")
        if self._mb is None or k > self.P2P_MAX_K:
            if exchange == "deferred":
                raise _lib.MdirError("exchange='deferred' needs the peer-memory mailboxes (and k <= %d)" % self.P2P_MAX_K)
            bits = torch.stack([local_status & STATUS_OVERFLOW, local_status & STATUS_UNCERTIFIED])
            if nq_all:
                self.dist.all_reduce(bits, op=self.dist.ReduceOp.MAX, group=self.group)      # per-bit MAX = OR over the ranks
            self._status = bits[0] | bits[1]
            return merge_keys(keys, self.world, self.group, k)
        if exchange == "deferred" and nq_all > self.P2P_MAX_Q:
            raise _lib.MdirError("exchange='deferred' handles at most %d queries per call" % self.P2P_MAX_Q)
        out_s = torch.empty((nq_all, k), dtype=torch.float32, device=self.device)
        out_i = torch.empty((nq_all, k), dtype=torch.int32, device=self.device)
        self._status = torch.empty((max(nq_all, 1),), dtype=torch.int32, device=self.device)[:nq_all]
        for q0 in range(0, nq_all, self.P2P_MAX_Q):
            q1 = min(q0 + self.P2P_MAX_Q, nq_all)
            self._exchange(keys[q0:q1], q1 - q0, k, 1 if exchange == "deferred" else 0, out_s[q0:q1], out_i[q0:q1],
                           local_status[q0:q1], self._status[q0:q1])
        return out_s, out_i

    def status(self):
        """Per-query status words of the step the last search()/drain() MERGED, OR-ed over the ranks (0 = exact and
        certified everywhere; bit 0 overflow, bit 1 uncertified on some rank, bit 2 a peer never arrived)."""
        return self._status

    def check_overflow(self):
        return bool(self._status.any().item())

    def search_collective_recovery(self, q, k, precision="fp32", shortlist=None):
        """The exact redo of a flagged batch, called by EVERY rank (the global status is identical on all of them):
        local search with recovery / widening, then the NCCL all-gather + merge route, which does not touch the
        mailboxes' sequence numbers and so may run between deferred steps."""
        s, i, keys = self.local.search(q, k, precision=precision, shortlist=shortlist, check=True, return_keys=True)
        if self.world == 1:
            return s, i
        return merge_keys(keys, self.world, self.group, k)

    def _exchange(self, keys, nq, k, mode, out_s, out_i, local_status=None, out_status=None):
        import ctypes as C
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().mdir_shard_exchange_merge(_lib.ptr(keys), nq, k, self._rank, self.world, self.P2P_MAX_Q, self.P2P_MAX_K, mode,
                                                            C.cast(self._mb, C.c_void_p), _lib.ptr(out_s), _lib.ptr(out_i),
                                                            _lib.ptr(local_status), _lib.ptr(out_status), _lib.stream()),
                       "mdir_shard_exchange_merge")

    def drain(self, n_q, k, out=None, status=None):
        """Merged result of the last exchange='deferred' call (every rank calls it; nothing is pushed).
        status: optional (n_q) int32 device tensor receiving that step's global status words."""
        if out is None:
            out = (torch.empty((n_q, k), dtype=torch.float32, device=self.device), torch.empty((n_q, k), dtype=torch.int32, device=self.device))
        if status is None:
            status = torch.empty((n_q,), dtype=torch.int32, device=self.device)
        self._status = status
        self._exchange(None, n_q, k, 2, out[0], out[1], None, status)
        return out


def merge_keys(local_keys, world, group, k):
    """All-gather (N_q, k) int64 keys from every rank and merge to the global top-k.
    Works on NCCL (device tensors) and gloo (host tensors; CPU tests of the sharding logic use
    merge_keys_host below instead of the CUDA merge)."""
    import torch.distributed as dist
    lib = _lib.lib()
    nq = local_keys.shape[0]
    gathered = torch.empty((world * nq, k), dtype=torch.int64, device=local_keys.device)
    dist.all_gather_into_tensor(gathered, local_keys.contiguous(), group=group)
    allk = gathered.view(world, nq, k).permute(1, 0, 2).contiguous().view(nq, world * k)
    cnt = torch.full((nq,), world * k, dtype=torch.int32, device=local_keys.device)
    out_s = torch.empty((nq, k), dtype=torch.float32, device=local_keys.device)
    out_i = torch.empty((nq, k), dtype=torch.int32, device=local_keys.device)
    with torch.cuda.device(local_keys.device):
        _lib.check(lib.mdir_topk_finalize(_lib.ptr(allk), world * k, _lib.ptr(cnt), 1, world * k, 0, nq, k, _lib.ptr(out_s), _lib.ptr(out_i),
                                          None, None, None, _lib.stream()), "mdir_topk_finalize")
    return out_s, out_i


# ---- host-side key helpers (pure integer logic; used by the gloo sharding tests) ------------

def make_keys_host(scores, idx):
    """numpy restatement of common.cuh:make_key for (score, index) arrays -> uint64 keys."""
    s = np.ascontiguousarray(scores, dtype=np.float32).copy()
    s[s == 0] = 0.0                                     # canonical +0
    u = s.view(np.uint32)
    o = np.where(u >> 31 != 0, ~u, u | np.uint32(0x80000000)).astype(np.uint32)
    d = np.where(np.isnan(s), np.uint32(0xffffffff), ~o).astype(np.uint32)      # NaN ranks last
    return (d.astype(np.uint64) << np.uint64(32)) | np.asarray(idx).astype(np.uint32).astype(np.uint64)


def keys_to_host(keys):
    """uint64 keys -> (scores fp32, idx int64); the all-ones key is padding (-inf, -1)."""
    keys = np.asarray(keys).astype(np.uint64)
    o = (~(keys >> np.uint64(32))).astype(np.uint32)
    u = np.where(o >> 31 != 0, o & np.uint32(0x7fffffff), ~o).astype(np.uint32)
    sc = u.view(np.float32).copy()
    idx = (keys & np.uint64(0xffffffff)).astype(np.int64)
    pad = keys == np.uint64(0xffffffffffffffff)
    sc[pad] = -np.inf
    idx[pad] = -1
    return sc, idx


def merge_keys_host(gathered, k):
    """gathered: (world, N_q, k) uint64 -> merged (N_q, k) uint64 (ascending key = best first)."""
    g = np.asarray(gathered).astype(np.uint64)
    world, nq, kk = g.shape
    allk = np.transpose(g, (1, 0, 2)).reshape(nq, world * kk)
    return np.sort(allk, axis=1)[:, :k]


def merge_keys_by_rank_host(gathered, k):
    """numpy restatement of the merge inside csrc/shard_merge.cu (pure integer logic, for the CPU tests): the world
    lists are sorted and their real keys unique, so the output slot of a key is its position in its own list plus,
    for every other list, the number of keys smaller than it (lower_bound); all-ones keys are padding."""
    g = np.asarray(gathered).astype(np.uint64)
    world, nq, kk = g.shape
    pad = np.uint64(0xffffffffffffffff)
    out = np.full((nq, k), pad, dtype=np.uint64)
    for q in range(nq):
        for r in range(world):
            for j in range(kk):
                key = g[r, q, j]
                if key == pad:
                    continue
                pos = j
                for o in range(world):
                    if o != r:
                        pos += int(np.searchsorted(g[o, q], key, side="left"))
                if pos < k:
                    out[q, pos] = key
    return out


class GraphedSearch:
    """One search step captured in a CUDA graph (CUDA streams and graphs instead of per-call
    launches): static query buffer in, static (scores, idx) out.  Works for an Index or a
    ShardedIndex (the NCCL all-gather of keys is captured too).  Every replay re-runs the whole
    chain: bf16 packing of the queries, sample scan, threshold select, filter scan, finalize,
    [fp32 re-scoring, finalize], [all-gather, merge].

        gs = GraphedSearch(index, n_q=70, k=100)
        scores, idx = gs(q)            # q: (70, D) fp32, host (pinned) or device
        gs.check_overflow()            # after a sync: True -> rerun through index.search()
    """

    def __init__(self, index, n_q, k, precision="fp32", shortlist=None, prof=None, deferred=False, overlap=False, split=False,
                 scan_ctas=0, fin_chunk=0, fin_stage=0):
        """deferred=True (ShardedIndex with peer-memory mailboxes): every replay pushes its keys and returns the merged
        result of the PREVIOUS replay (see ShardedIndex.search); drain() returns the last one.
        overlap=True (same precondition): the graph holds only the LOCAL part of the step (pack, scan, finalize -> this
        shard's sorted keys); exchange() launches the NVLink push + merge kernel for those keys on whatever stream is
        current -- a side stream in SearchPipeline, so that the exchange of step t runs while the scan of step t+1
        streams the shard (the scan grid leaves SMs free for it) and its latency leaves the step's critical path."""
        self.index = index
        self.local = index.local if isinstance(index, ShardedIndex) else index
        dev = self.local.device
        self.n_q, self.k, self.precision, self.shortlist = int(n_q), int(k), precision, shortlist
        sharded = isinstance(index, ShardedIndex) and index.world > 1
        self._has_exchange = sharded
        self.overlap = bool(overlap) and sharded and index._mb is not None and self.k <= index.P2P_MAX_K and self.n_q <= index.P2P_MAX_Q
        self.deferred = bool(deferred) and sharded and not self.overlap
        self.q = torch.zeros((n_q, self.local.D), dtype=torch.float32, device=dev)
        self.local.prof = None
        extra = {"exchange": "deferred"} if self.deferred else {}
        # split=True (overlap mode, one-launch scan route, fp32): TWO graphs with a private candidate workspace --
        # `graph` = pack + scan, `back` = finalize + certified re-score -- so that the pipeline can run the finalize (and
        # the exchange) of ticket t on the side stream while the compute stream scans ticket t+1
        k_eff = min(self.k, self.local.n)
        self.kth = max(k_eff, min(self.local.n, int(shortlist or default_shortlist(self.k))))
        self.split = (bool(split) and (self.overlap or (bool(overlap) and not sharded)) and precision == "fp32" and self.local.db32 is not None
                      and k_eff == self.k and self.n_q <= MAX_Q and self.local._fused_ok(self.kth, self.n_q))
        if self.split and not sharded:
            self.overlap = True                  # a single GPU: no exchange, but the finalize half still runs on the side stream
        # SM partition of the split mode: the scan's persistent grid capped at scan_ctas (0 = all SMs), finalize launched
        # in slices of fin_chunk queries on single CTAs (0 = one launch, 2-CTA clusters) -- together at most 148 SMs, so
        # that the side stream's finalize finds room while the compute stream scans
        self.scan_ctas, self.fin_chunk, self.fin_stage = int(scan_ctas), int(fin_chunk), int(fin_stage)
        if self.split:
            self._init_split(prof)
            return

        def step():
            if self.overlap:
                return self.local.search(self.q, self.k, precision=self.precision, shortlist=self.shortlist, check=False, return_keys=True)
            return index.search(self.q, self.k, precision=self.precision, shortlist=self.shortlist, check=False, **extra)

        with torch.cuda.device(dev):
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):                      # warm-up: workspaces, function attributes, NCCL channels
                    step()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            self.local.prof = prof
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                res = step()
                self.ovf = self.local._ovf[:n_q].clone()      # this graph's own copy of the LOCAL status words of this step
                if self.overlap:
                    self.keys = res[2]
                    self.out = (torch.empty((n_q, self.k), dtype=torch.float32, device=dev), torch.empty((n_q, self.k), dtype=torch.int32, device=dev))
                    self.status = torch.zeros((n_q,), dtype=torch.int32, device=dev)
                else:
                    self.out = res
                    # status words of the step whose result `out` holds: the world's OR for a sharded index (in deferred
                    # mode that is the previous step, like `out`)
                    self.status = index._status[:n_q].clone() if sharded else self.ovf
            self.local.prof = None
            if self.overlap:
                self.local_done, self.done = torch.cuda.Event(), torch.cuda.Event()

    def _init_split(self, prof):
        loc, dev, nq, k = self.local, self.local.device, self.n_q, self.k
        lib = _lib.lib()
        loc._ws_tag = ("graph", id(self))
        try:
            tau, cand, cnt = loc._cand_bufs(nq)
            ovf = loc._buf("ovf", (max(nq, 1),), torch.int32)
        finally:
            loc._ws_tag = None
        ws = loc._fused_ws()
        i8 = loc._i8_route(self.kth, nq)         # the same route choice as Index.search
        if i8:
            stats = loc.stats()
            self.q8 = torch.empty((2 * (-(-nq // 16) * 16), loc.D), dtype=torch.int8, device=dev)
            self.q8_scale = torch.empty((nq, 2), dtype=torch.float32, device=dev)
            self.q8_eps = torch.empty((nq,), dtype=torch.float32, device=dev)
        else:
            self.q16 = torch.empty((nq, loc.D), dtype=torch.bfloat16, device=dev)
        self.keys = torch.empty((nq, k), dtype=torch.int64, device=dev)
        self.local_out = (torch.empty((nq, k), dtype=torch.float32, device=dev), torch.empty((nq, k), dtype=torch.int32, device=dev))
        self.ovf = ovf[:nq]
        if self._has_exchange:
            self.out = (torch.empty((nq, k), dtype=torch.float32, device=dev), torch.empty((nq, k), dtype=torch.int32, device=dev))
            self.status = torch.zeros((nq,), dtype=torch.int32, device=dev)
        else:
            self.out, self.status = self.local_out, self.ovf

        def front():
            if i8:
                _lib.check(lib.mdir_pack_q_i8(_lib.ptr(self.q), nq, loc.D, _lib.ptr(stats), _lib.ptr(self.q8), _lib.ptr(self.q8_scale),
                                              _lib.ptr(self.q8_eps), _lib.stream()), "mdir_pack_q_i8")
            else:
                _lib.check(lib.mdir_pack_bf16(_lib.ptr(self.q), nq, loc.D, 0, _lib.ptr(self.q16), _lib.stream()), "mdir_pack_bf16")
            if prof is not None:
                prof.begin()
            lib.mdir_tune(1, self.scan_ctas)
            try:
                if i8:
                    _lib.check(lib.mdir_sim_scan_fused_i8(_lib.ptr(loc.db8), _lib.ptr(loc.row_scale), loc.n, _lib.ptr(self.q8), _lib.ptr(self.q8_scale),
                                                          nq, loc.D, self.kth, _lib.ptr(tau), loc.idx_base, _lib.ptr(cand), _lib.ptr(cnt), 0,
                                                          FUSED_CAP_L, _lib.ptr(ws), _lib.stream()), "mdir_sim_scan_fused_i8")
                else:
                    _lib.check(lib.mdir_sim_scan_fused_bf16(_lib.ptr(loc.db16), loc.n, _lib.ptr(self.q16), nq, loc.D, self.kth, _lib.ptr(tau),
                                                            loc.idx_base, _lib.ptr(cand), _lib.ptr(cnt), 0, FUSED_CAP_L, _lib.ptr(ws),
                                                            _lib.stream()), "mdir_sim_scan_fused_bf16")
            finally:
                lib.mdir_tune(1, 0)
            if prof is not None:
                prof.end(loc.n * loc.D + 4 * loc.n if i8 else loc.n * loc.D * 2)

        def back():
            chunk = self.fin_chunk if self.fin_chunk > 0 else nq
            lib.mdir_tune(2, 0 if self.fin_chunk > 0 else 1)
            lib.mdir_tune(3, self.fin_stage)
            try:
                for q0 in range(0, nq, chunk):
                    q1 = min(q0 + chunk, nq)
                    loc._finalize(cand[q0:q1], cnt[q0:q1], q1 - q0, self.kth, self.local_out[0][q0:q1], self.local_out[1][q0:q1],
                                  self.keys[q0:q1], tau[q0:q1], self.ovf[q0:q1], (self.q[q0:q1], k), caps=(0, FUSED_CAP_L),
                                  q_eps=self.q8_eps[q0:q1] if i8 else None)
            finally:
                lib.mdir_tune(2, 1)
                lib.mdir_tune(3, 0)
            if self._has_exchange:
                # the NVLink push + merge of these keys rides in the same graph: one launch per ticket on the side stream
                self.index._exchange(self.keys, nq, k, 0, self.out[0], self.out[1], self.ovf, self.status)

        with torch.cuda.device(dev):
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(2):
                    front()
                    back()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            self.graph, self.back = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                front()
            with torch.cuda.graph(self.back):
                back()
            self.local_done, self.done = torch.cuda.Event(), torch.cuda.Event()

    def exchange(self):
        """overlap mode: push this graph's keys to every peer and merge the world's (synchronous exchange of THIS step) on
        the current stream, into `out` / `status`.  Every rank calls it once per replay, in the same order."""
        if getattr(self, "split", False):
            self.back.replay()                   # finalize + certified re-score (+ exchange and merge) of this graph's scan
            return
        if self._has_exchange:
            self.index._exchange(self.keys, self.n_q, self.k, 0, self.out[0], self.out[1], self.ovf, self.status)

    def __call__(self, q=None):
        if q is not None:
            self.q.copy_(q, non_blocking=True)
        self.graph.replay()
        if self.overlap:
            self.exchange()
        return self.out

    def drain(self):
        """deferred mode: the merged result of the last replay, written into this graph's static outputs."""
        if self.deferred:
            self.index.drain(self.n_q, self.k, out=self.out, status=self.status)
        return self.out

    def check_overflow(self):
        """True when some query of the step `out` holds was flagged (overflow / uncertified shortlist, on any rank):
        rerun that batch through index.search() (ShardedIndex: search_collective_recovery on every rank)."""
        return bool(self.status.any().item())


class SearchPipeline:
    """Host-facing serving loop: query batches arrive in (pinned) host memory, results go back to
    pinned host memory, and the copies of one step overlap the scan of its neighbours.

        pipe = SearchPipeline(index, n_q=70, k=100)            # Index or ShardedIndex
        t0 = pipe.submit(q_host_0)                             # H2D -> graph replay -> D2H, all asynchronous
        t1 = pipe.submit(q_host_1)
        scores, idx = pipe.result(t0)                          # numpy views of pinned buffers, valid until
        ...                                                    # `depth` more submits

    `depth` CUDA graphs (one static query buffer and output set each) replay back to back on one
    compute stream; uploads and downloads run on their own streams, ordered by events only.  A step
    whose candidate lists overflowed is transparently redone through index.search() (exact recovery).
    With a ShardedIndex every rank must submit the same sequence (the all-gather is inside the graphs)."""

    def __init__(self, index, n_q, k, depth=None, precision="fp32", shortlist=None, prof=None, deferred=None, overlap=None, split=True,
                 scan_ctas=None):
        """overlap (default: on for a ShardedIndex with peer-memory mailboxes): the graphs hold the local part of a step;
        the NVLink exchange + merge of step t runs on its own stream while the compute stream already scans step t+1
        (GraphedSearch(overlap=True)) -- results are those of the SAME ticket, nothing lags.
        deferred (the earlier scheme, kept selectable): the merge of step t runs inside the replay of step t+1 (or in a
        drain when nothing follows).  depth = steps in flight (default 2; 3 for the two sharded schemes)."""
        self.index = index
        self.local = index.local if isinstance(index, ShardedIndex) else index
        dev = self.local.device
        self.n_q, self.k = int(n_q), int(k)
        self.precision, self.shortlist = precision, shortlist
        sharded = isinstance(index, ShardedIndex) and index.world > 1
        p2p_ok = sharded and index._mb is not None and self.k <= index.P2P_MAX_K and self.n_q <= index.P2P_MAX_Q
        if overlap is None:
            overlap = p2p_ok and not deferred
        self.overlap = bool(overlap) and p2p_ok
        if deferred is None:
            deferred = False
        self.deferred = bool(deferred) and p2p_ok and not self.overlap
        # a single GPU has no exchange, but the split graphs still move finalize + re-score of ticket t beside the scan of
        # ticket t+1: the scan's persistent grid is capped (SINGLE_GPU_SCAN_CTAS of 148 SMs; the stream stays HBM-bound)
        # so that the finalize CTAs find SMs
        # -- measured on the R1M shape: 660 us per step as one graph, 664-705 us split (tools/time_split_1gpu.py): the capped
        # scan loses what the hidden finalize gains, so this stays opt-in (split="single")
        single_split = (not sharded) and split == "single" and overlap is not False and not deferred
        if scan_ctas is None:
            scan_ctas = SINGLE_GPU_SCAN_CTAS if single_split else 0
        n_graphs = int(depth) if depth else (3 if (self.deferred or self.overlap or single_split) else 2)
        self.graphs = [GraphedSearch(index, n_q, k, precision=precision, shortlist=shortlist, prof=prof if s == 0 else None,
                                     deferred=self.deferred, overlap=self.overlap or single_split, split=split, scan_ctas=scan_ctas)
                       for s in range(n_graphs)]
        if single_split:
            self.overlap = all(g.split for g in self.graphs)
        self.depth = n_graphs
        with torch.cuda.device(dev):
            self.compute, self.h2d, self.d2h, self.exch = (torch.cuda.Stream(device=dev) for _ in range(4))
            self.slots = []
            for _ in range(self.depth):
                self.slots.append({
                    "scores": torch.empty((self.n_q, self.k), dtype=torch.float32).pin_memory(),
                    "idx": torch.empty((self.n_q, self.k), dtype=torch.int32).pin_memory(),
                    "ovf": torch.zeros((self.n_q,), dtype=torch.int32).pin_memory(),
                    "up": torch.cuda.Event(), "done": torch.cuda.Event(), "down": torch.cuda.Event(), "local": torch.cuda.Event(),
                    "q": None, "pending": False, "merged": False, "used": False})
            if self.deferred:
                self.drain_out = (torch.empty((self.n_q, self.k), dtype=torch.float32, device=dev),
                                  torch.empty((self.n_q, self.k), dtype=torch.int32, device=dev))
                self.drain_status = torch.zeros((self.n_q,), dtype=torch.int32, device=dev)
                with torch.cuda.stream(self.compute):          # forget the graphs' warm-up pushes
                    index.drain(self.n_q, self.k, out=self.drain_out, status=self.drain_status)
            torch.cuda.synchronize(dev)
        self.n_submitted = 0
        self.n_recovered = 0          # steps redone exactly because a status word was raised

    def _download(self, slot, src, status):
        """Queue the D2H of a merged result and its status words into `slot`'s pinned buffers (ordered after the compute
        stream's last event)."""
        with torch.cuda.stream(self.d2h):
            slot["scores"].copy_(src[0], non_blocking=True)
            slot["idx"].copy_(src[1], non_blocking=True)
            slot["ovf"].copy_(status, non_blocking=True)
            slot["down"].record()
        slot["merged"] = True

    def submit(self, q):
        """q: (n_q, D) fp32, pinned host memory for a truly asynchronous upload (device tensors work too).
        Returns a ticket for result().  The caller keeps q unchanged until result(ticket) returned."""
        t_new = self.n_submitted
        slot, gs = self.slots[t_new % self.depth], self.graphs[t_new % self.depth]
        if slot["pending"]:
            raise _lib.MdirError("SearchPipeline: collect result() of ticket %d before submitting more" % (t_new - self.depth))
        q = torch.as_tensor(q)
        if tuple(q.shape) != tuple(gs.q.shape):
            raise _lib.MdirError("SearchPipeline expects query batches of shape %s" % (tuple(gs.q.shape),))
        with torch.cuda.stream(self.h2d):
            gs.q.copy_(q, non_blocking=True)            # this slot's previous replay was drained by result()
            slot["up"].record()
        with torch.cuda.stream(self.compute):
            self.compute.wait_event(slot["up"])
            if self.overlap and slot["used"]:
                self.compute.wait_event(slot["done"])      # this graph's key buffer: its previous exchange has read it
            gs.graph.replay()
            if self.overlap:
                slot["local"].record()
            else:
                slot["done"].record()
        if self.overlap:
            with torch.cuda.stream(self.exch):             # exchange + merge of THIS ticket, behind the next ticket's scan
                self.exch.wait_event(slot["local"])
                gs.exchange()
                slot["done"].record()
        slot["q"], slot["pending"], slot["merged"], slot["used"] = q, True, False, True
        self.d2h.wait_event(slot["done"])
        if not self.deferred:
            self._download(slot, gs.out, gs.status)
        elif t_new >= 1 and self.slots[(t_new - 1) % self.depth]["pending"]:
            self._download(self.slots[(t_new - 1) % self.depth], gs.out, gs.status)        # this replay merged the previous ticket
        self.n_submitted += 1
        return t_new

    def result(self, ticket):
        """Blocks until step `ticket` is in host memory; returns (scores (n_q, k) fp32, idx (n_q, k) int32) numpy views."""
        if not (self.n_submitted - self.depth <= ticket < self.n_submitted):
            raise _lib.MdirError("SearchPipeline: ticket %d is not in flight" % ticket)
        slot = self.slots[ticket % self.depth]
        if not slot["pending"]:
            raise _lib.MdirError("SearchPipeline: result(%d) was already collected" % ticket)
        if not slot["merged"]:
            # deferred exchange and nothing was submitted after this ticket: merge it now (every rank does the same)
            if ticket != self.n_submitted - 1:
                raise _lib.MdirError("SearchPipeline: collect deferred results in submission order")
            with torch.cuda.stream(self.compute):
                self.index.drain(self.n_q, self.k, out=self.drain_out, status=self.drain_status)
                ev = torch.cuda.Event()
                ev.record()
            self.d2h.wait_event(ev)
            self._download(slot, self.drain_out, self.drain_status)
        slot["down"].synchronize()
        slot["pending"] = False
        if bool(slot["ovf"].any()):
            # some query of this step was flagged (candidate overflow or a failed shortlist certificate; for a sharded
            # index on ANY rank -- the status words are the world's OR, so every rank takes this branch together)
            self.n_recovered += 1
            sharded = isinstance(self.index, ShardedIndex) and self.index.world > 1
            if sharded and bool((slot["ovf"] & STATUS_PEER_TIMEOUT).any()):
                raise _lib.MdirError("SearchPipeline: a peer rank did not deliver its keys for ticket %d within the bounded wait" % ticket)
            # exact recovery, ordered after everything already queued on the compute stream (shared workspaces)
            if self.overlap:
                self.compute.wait_stream(self.exch)
            with torch.cuda.stream(self.compute):
                if sharded:
                    s, i = self.index.search_collective_recovery(slot["q"], self.k, precision=self.precision, shortlist=self.shortlist)
                else:
                    s, i = self.index.search(slot["q"], self.k, precision=self.precision, shortlist=self.shortlist)
                slot["scores"].copy_(s)
                slot["idx"].copy_(i)
            self.compute.synchronize()
        slot["q"] = None
        return slot["scores"].numpy(), slot["idx"].numpy()

    def map(self, batches):
        """Generator over an iterable of query batches, keeping `depth` steps in flight."""
        tickets = []
        for q in batches:
            if len(tickets) == self.depth:
                yield self.result(tickets.pop(0))
            tickets.append(self.submit(q))
        for t in tickets:
            yield self.result(t)
