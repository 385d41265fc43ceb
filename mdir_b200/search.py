"""Query x database similarity, top-k and full ranks.

Replaces, for mdir's evaluation (mdir/components/optim/score/cirscore.py:65-70):

    scores = np.dot(vecs.T, qvecs)          # (N_db, N_q)
    ranks  = np.argsort(-scores, axis=0)    # (N_db, N_q) int64

* ``rank(vecs, qvecs)``      -- the drop-in: host (D,N) matrices in, (N_db,N_q) int64 ranks out.
* ``Index``                  -- a database resident in HBM as row-major bf16 (+ optional fp32
                                master for exact re-scoring); ``search`` = tcgen05 scan with the
                                top-k selection fused into the epilogue, ``scores`` / ``ranks``
                                = the dense path.  Rows can be removed, restored and appended in
                                place (``remove`` / ``restore`` / ``add``: a live-row bitmap the
                                scan reads); ``compact`` purges removed rows and shrinks the scan to the
                                live ones, ids unchanged.  ``range_search`` = every live row whose
                                score reaches a per-query threshold (CSR output, exact fp32).
* ``ShardedIndex``           -- rows sharded contiguously over the ranks of a torch.distributed
                                group; local top-k + one all-gather of N_q*k keys + merge.
* ``ranks_from_scores`` / ``topk_from_scores`` -- the sort/selection kernels fed an existing
                                (N_db, N_q) score matrix (bit-exact vs the stable argsort).
"""
import contextlib
import ctypes as C
import functools

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
DENSE_ROUTE = (0, 0, 0)   # Index._route's (route, n_sample, stride) of the dense route


STATUS_OVERFLOW, STATUS_UNCERTIFIED, STATUS_PEER_TIMEOUT = 1, 2, 4     # MDIR_STATUS_* (+ the exchange's own bit)
STATUS_RANGE_FULL = 8     # MDIR_STATUS_RANGE_FULL: a captured range step found more survivors than max_results
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
# range_search: initial capacity of each scan CTA's candidate segment.  At 10,000 fp32 matches per query in 1 M rows the
# scan passes ~14,000 candidates (the certified bound lowers its threshold), ~92 per segment on average; a block whose
# segments still overflow is re-scanned once at the exact capacity the counts report.
RANGE_CAP_L = 192
RANGE_CHUNK = 1024      # MDIR_RANGE_CHUNK: candidate slots per CTA of mdir_range_gather
RANGE_STAGE = 16384     # survivors of one query that mdir_range_emit sorts in shared memory; more take the group merge
# bytes of candidate + survivor keys (8 B each, 148 * cap_l + chunks * RANGE_CHUNK per query) one re-scan may hold: a
# block whose exact counts need more is re-scanned in smaller query groups (min_score = -inf over 1 M rows needs ~16 MB
# per query, so 32 queries per group)
RANGE_BUDGET = 1 << 29


def default_shortlist(k):
    """Initial bf16 shortlist for an exact fp32 top-k: 1.25 k rounded up to a multiple of 64 (whole rounds of the
    2 x 32 re-scoring warps).  It only has to be a good first guess: the finalize kernel extends it with every
    candidate whose bf16 score is within the certified error bound of the k-th fp32 score, and flags the query
    when even the candidate list is not provably deep enough (mdir_topk_finalize_rescore)."""
    return -(-(-(-5 * int(k) // 4)) // 64) * 64


@functools.lru_cache(maxsize=4096)
def topk_plan(n_db, kth, sm_count):
    """mdir_topk_plan: (route, n_sample, stride) of a top-k over n_db rows at selection depth kth on sm_count SMs (the
    rules live in composite.cu only; see Index._route).  Host-only: no CUDA call; cached, so that eager search() pays
    no ctypes call per block."""
    route, n_sample, stride = C.c_int(), C.c_int(), C.c_int()
    _lib.check(_lib.lib().mdir_topk_plan(int(n_db), int(kth), int(sm_count), C.byref(route), C.byref(n_sample), C.byref(stride)),
               "mdir_topk_plan")
    return route.value, n_sample.value, stride.value


def _as_dev_f32(x, device):
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    if x.dtype != torch.float32:
        x = x.float()
    if x.device != device:
        x = x.pin_memory().to(device, non_blocking=True) if x.device.type == "cpu" else x.to(device)
    return x.contiguous()


def pack_bf16(x, dxn=False, out=None):
    """x fp32 cuda: (n, D) rows, or with dxn=True the reference's (D, n) -> (n, D) bf16 rows.
    out: the first n rows of a preallocated contiguous (>= n, D) bf16 tensor to write (default: a new one)."""
    _lib.require_cuda(x, "descriptors")
    x = x.contiguous()
    if dxn:
        D, n = x.shape
    else:
        n, D = x.shape
    if D % 8:
        raise _lib.MdirError("descriptor dimension must be a multiple of 8 (got %d)" % D)
    if out is None:
        out = torch.empty((n, D), dtype=torch.bfloat16, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().mdir_pack_bf16(_lib.ptr(x), n, D, 1 if dxn else 0, _lib.ptr(out), _lib.stream()), "mdir_pack_bf16")
    return out


def check_ids(ids, lo, hi):
    """ids (host or device tensor, numpy array or sequence of integers) -> int64 numpy rows ids - lo; MdirError when
    an id lies outside [lo, hi).  The host-side validation of Index.remove / restore."""
    if isinstance(ids, torch.Tensor):
        ids = ids.detach().cpu().numpy()
    a = np.asarray(ids)
    if a.size and not np.issubdtype(a.dtype, np.integer):
        raise _lib.MdirError("ids must be integers (got %s)" % a.dtype)
    a = a.astype(np.int64).ravel()
    bad = (a < lo) | (a >= hi)
    if bad.any():
        raise _lib.MdirError("id %d is outside this index's ids [%d, %d)" % (int(a[bad][0]), lo, hi))
    return a - lo


def compaction_schedule(live, chunk):
    """The in-place move of Index.compact: live (bool per used slot) -> [(lo, hi, dst0, n_dst, staged)], chunks of at most
    `chunk` slots in ascending order from the first dead slot.  The n_dst live slots of [lo, hi) go, in order, to
    [dst0, dst0 + n_dst); dst0 = live slots before lo, so a chunk only overwrites slots below hi, which this or an
    earlier chunk has already read.  staged = the destinations reach into the chunk itself (dst0 + n_dst > lo): its
    rows are gathered into scratch first; otherwise reads and writes are disjoint and the chunk moves directly."""
    live = np.asarray(live, dtype=bool)
    dead = np.flatnonzero(~live)
    if dead.size == 0:
        return []
    cum = np.concatenate([[0], np.cumsum(live, dtype=np.int64)])
    out = []
    for lo in range(int(dead[0]), live.size, int(chunk)):
        hi = min(lo + int(chunk), live.size)
        dst0, n_dst = int(cum[lo]), int(cum[hi] - cum[lo])
        if n_dst:
            out.append((lo, hi, dst0, n_dst, dst0 + n_dst > lo))
    return out


def range_thresholds(min_score, nq):
    """min_score (a float, or one per query: tensor / array / sequence of nq) -> (nq,) float32 numpy.  A float64 value is
    rounded UP to float32, so that an fp32 score passes the float32 threshold exactly when it is >= the value given.
    MdirError on NaN or a wrong length."""
    if isinstance(min_score, torch.Tensor):
        min_score = min_score.detach().cpu().numpy()
    a = np.asarray(min_score, dtype=np.float64)
    if a.ndim == 0:
        a = np.full((nq,), float(a))
    if a.shape != (nq,):
        raise _lib.MdirError("min_score must be a float or hold one value per query (%d), got shape %s" % (nq, a.shape))
    if np.isnan(a).any():
        raise _lib.MdirError("min_score is NaN for query %d" % int(np.flatnonzero(np.isnan(a))[0]))
    a32 = a.astype(np.float32)
    low = a32.astype(np.float64) < a
    a32[low] = np.nextafter(a32[low], np.float32(np.inf))
    return a32


def range_chunks(cap_l):
    """mdir_range_chunks: gather chunks covering one candidate row of 148 segments of cap_l keys."""
    return -(-148 * int(cap_l) // RANGE_CHUNK)


def range_csr(run_len):
    """run_len (nq, n_chunks): survivors of every gather chunk -> (counts (nq,) int64, lims (nq + 1,) int64 -- the CSR
    offsets, query i at [lims[i], lims[i + 1]) --, run_off (nq, n_chunks) int32: survivors of the query before chunk c)."""
    run_len = np.asarray(run_len, dtype=np.int64)
    counts = run_len.sum(axis=1)
    lims = np.zeros((run_len.shape[0] + 1,), dtype=np.int64)
    np.cumsum(counts, out=lims[1:])
    run_off = np.ascontiguousarray(np.cumsum(run_len, axis=1) - run_len, dtype=np.int32)
    return counts, lims, run_off


def range_rescan_plan(max_seg, budget=RANGE_BUDGET):
    """After a range scan overflowed: (cap_l, group) = the segment capacity that holds the largest count any segment
    reported (rounded up to 32), and how many queries one re-scan takes so that its candidate + survivor keys stay
    within `budget` bytes (at least one)."""
    max_seg = np.asarray(max_seg, dtype=np.int64)
    cap = max(32, -(-int(max_seg.max()) // 32) * 32)
    per_query = 8 * (148 * cap + range_chunks(cap) * RANGE_CHUNK)
    return cap, int(max(1, min(max_seg.size, budget // per_query)))


def range_stage_cap(max_results):
    """mdir_range_emit's stage_cap for a captured range step: max_results rounded up to a power of two, at least 32."""
    stage = 32
    while stage < int(max_results):
        stage *= 2
    return stage


def range_splice(lims, scores, ids, flagged, sub_lims, sub_scores, sub_ids):
    """Replace the results of the queries `flagged` (ascending query numbers) in the CSR (lims, scores, ids) by the CSR
    (sub_lims, sub_scores, sub_ids) of those queries, in the same order -> a new packed CSR (lims, scores, ids), numpy.
    RangePipeline's recovery: the flagged queries of a captured step redone by Index.range_search."""
    lims, sub_lims = np.asarray(lims, dtype=np.int64), np.asarray(sub_lims, dtype=np.int64)
    flagged = np.asarray(flagged, dtype=np.int64).ravel()
    nq = lims.size - 1
    if flagged.size and (flagged[0] < 0 or flagged[-1] >= nq or (np.diff(flagged) <= 0).any()):
        raise _lib.MdirError("range_splice: flagged must be ascending query numbers in [0, %d)" % nq)
    if sub_lims.size != flagged.size + 1:
        raise _lib.MdirError("range_splice: %d flagged queries need %d sub_lims, got %d" % (flagged.size, flagged.size + 1, sub_lims.size))
    sub_of = np.full((nq,), -1, dtype=np.int64)
    sub_of[flagged] = np.arange(flagged.size)
    counts = np.diff(lims)
    counts[flagged] = np.diff(sub_lims)
    out_lims = np.zeros((nq + 1,), dtype=np.int64)
    np.cumsum(counts, out=out_lims[1:])
    out_s = np.empty((int(out_lims[-1]),), dtype=np.asarray(scores).dtype)
    out_i = np.empty((int(out_lims[-1]),), dtype=np.asarray(ids).dtype)
    for j in range(nq):
        a, b = out_lims[j], out_lims[j + 1]
        if sub_of[j] < 0:
            out_s[a:b], out_i[a:b] = scores[lims[j]:lims[j + 1]], ids[lims[j]:lims[j + 1]]
        else:
            k = sub_of[j]
            out_s[a:b], out_i[a:b] = sub_scores[sub_lims[k]:sub_lims[k + 1]], sub_ids[sub_lims[k]:sub_lims[k + 1]]
    return out_lims, out_s, out_i


def ids_for_rank(ids, ranges, rank):
    """Global ids -> the int64 numpy ids that rank `rank` owns, ranges[r] = (first id, end id) of rank r (see
    ShardedIndex.shard_bounds).  MdirError when an id lies in no rank's range."""
    if isinstance(ids, torch.Tensor):
        ids = ids.detach().cpu().numpy()
    a = np.asarray(ids)
    if a.size and not np.issubdtype(a.dtype, np.integer):
        raise _lib.MdirError("ids must be integers (got %s)" % a.dtype)
    a = a.astype(np.int64).ravel()
    owned = np.zeros(a.shape, dtype=bool)
    for lo, hi in ranges:
        owned |= (a >= lo) & (a < hi)
    if not owned.all():
        raise _lib.MdirError("id %d is outside every shard of this index" % int(a[~owned][0]))
    lo, hi = ranges[rank]
    return a[(a >= lo) & (a < hi)]


class Index:
    """A (shard of a) descriptor database on one GPU.

    Mutable in place: ``remove(ids)`` hides rows from every later search, ``restore(ids)`` undoes that, and
    ``add(vecs)`` writes new rows into free slots of a ``capacity`` larger than the initial database.  An id names
    one row for the life of the index and is never reused; until the first ``compact()`` it is idx_base + slot.
    Which rows are live is one bitmap on the device (1 bit per slot) that every top-k route reads in the scan
    epilogue.  The scan covers the used slots [0, n_used), a device-side extent: removed rows cost scan bandwidth like
    live ones until ``compact()`` moves the live rows to the front (stably), purges the removed ones and shrinks the
    extent; a slot -> id map keeps the ids.  CUDA graphs captured over the index see every later mutation and
    compaction without re-capture."""

    fused = True      # allow the one-launch threshold + filter route (False: always sample -> select -> filter)
    compact_chunk = 16384   # slots per chunk of compact()'s in-place move (its scratch holds one chunk's live rows)
    certify = True    # precision="fp32": prove the shortlist complete (status bit 2 + widening when it cannot be)
    tiered = True     # int8 route: screen the certified extension on the bf16 rows before the fp32 gather (same output)
    _sms = None
    _mutations = 0    # remove / restore / add / compact calls that changed the index (Diffusion's graph goes stale)

    def __init__(self, vecs, dxn=False, device="cuda", keep_fp32=True, idx_base=0, capacity=None):
        """vecs: (n, D) fp32 rows (torch/numpy, host or device), or (D, n) with dxn=True
        (the layout extract_vectors returns, cirtorch/networks/imageretrievalnet.py:291).
        capacity (default n): slots allocated for rows; add() fills slots n, n + 1, ...  With capacity > n the bf16
        rows, the fp32 master (a copy of vecs) and, once built, the int8 plane are allocated at capacity, the free
        slots zero.  The scan covers the filled slots.  idx_base + capacity must stay <= 2**32."""
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.MdirError("Index needs a CUDA device (no CPU path)")
        v = _as_dev_f32(vecs, self.device)
        n, D = (v.shape[1], v.shape[0]) if dxn else (v.shape[0], v.shape[1])
        cap = n if capacity is None else int(capacity)
        if cap < n:
            raise _lib.MdirError("capacity %d is smaller than the %d rows given" % (cap, n))
        if int(idx_base) < 0 or int(idx_base) + cap > 1 << 32:
            raise _lib.MdirError("idx_base + capacity must stay within [0, 2**32]")
        with torch.cuda.device(self.device):
            db16 = torch.zeros((cap, D), dtype=torch.bfloat16, device=self.device) if cap > n else None
            self.db16 = pack_bf16(v, dxn=dxn, out=db16)
            self.n, self.D = self.db16.shape
            self.idx_base = int(idx_base)
            self.db32 = None
            if keep_fp32:
                if cap == n:
                    self.db32 = v.t().contiguous() if dxn else v
                else:
                    self.db32 = torch.zeros((cap, D), dtype=torch.float32, device=self.device)
                    self.db32[:n].copy_(v.t() if dxn else v)
            self._init_live(n)
        self._ws = {}
        self._stats = None
        self.db8 = self.row_scale = None
        self.route = None
        self.cert = {"queries": 0, "flagged": 0, "widened_blocks": 0, "uncertified": 0, "int8_blocks": 0, "int8_redone": 0}
        self.range_stats = {"queries": 0, "blocks": 0, "rescans": 0, "rescan_groups": 0, "large_sorts": 0}

    @classmethod
    def from_packed(cls, db16, db32=None, idx_base=0):
        self = cls.__new__(cls)
        self.device = db16.device
        self.db16 = db16
        self.n, self.D = db16.shape
        self.db32 = db32
        self.idx_base = int(idx_base)
        with torch.cuda.device(self.device):
            self._init_live(self.n)
        self._ws = {}
        self._stats = None
        self.db8 = self.row_scale = None
        self.route = None
        self.cert = {"queries": 0, "flagged": 0, "widened_blocks": 0, "uncertified": 0, "int8_blocks": 0, "int8_redone": 0}
        self.range_stats = {"queries": 0, "blocks": 0, "rescans": 0, "rescan_groups": 0, "large_sorts": 0}
        return self

    # ------------------------------------------------------------------ live rows
    def _init_live(self, n_used):
        """The live bitmap: bit s & 31 of word s >> 5 = slot s is live; ones for the n_used filled slots, zeros for the
        free tail.  It covers whole 256-row scan tiles (the select kernel reads the words of a sample's last tile past
        the end) and is modified only in place, so a captured graph keeps reading the current version."""
        words = -(-self.n // TILE) * (TILE // 32)
        bits = np.zeros(words * 32, dtype=bool)
        bits[:n_used] = True
        host = np.packbits(bits, bitorder="little").view("<u4").view(np.int32)
        self.live = torch.from_numpy(host.copy()).to(self.device)
        self._live_host = bits[:self.n].copy()     # host mirror: id validation and n_live without a device read-back
        self._n_used = int(n_used)
        # the scan extent (slots [0, n_used) are scanned) and the slot -> id map (uint32 ids, identity until compact()),
        # both on the device for the kernels and captured graphs, updated in place in stream order
        self.n_scan = torch.tensor([self._n_used], dtype=torch.int64, device=self.device)
        ident = np.arange(self.idx_base, self.idx_base + self.n, dtype=np.int64)
        self.slot_id = torch.from_numpy(ident.astype(np.uint32).view(np.int32)).to(self.device)
        self._ids = ident[:self._n_used].copy()    # host mirror over the used slots, strictly increasing
        self._next_id = self._n_used               # ids idx_base .. idx_base + _next_id - 1 have been issued

    @property
    def n_live(self):
        """Number of live rows (filled and not removed)."""
        return int(self._live_host.sum())

    def _require_all_live(self, what):
        if self.n_live != self.n:
            raise _lib.MdirError("%s scores every slot and does not support an index with removed rows or free capacity "
                                 "(%d of %d slots live); use search()" % (what, self.n_live, self.n))

    def _set_live(self, rows, value):
        rows = np.unique(rows)
        rows = rows[self._live_host[rows] != bool(value)]          # repeated and no-op ids cost nothing
        if rows.size == 0:
            return
        self._mutations += 1
        ids = torch.from_numpy(rows + self.idx_base).to(self.device)
        _lib.check(_lib.lib().mdir_live_update(_lib.ptr(self.live), self.n, self.idx_base, _lib.ptr(ids), int(rows.size), int(value),
                                               _lib.stream()), "mdir_live_update")
        self._live_host[rows] = bool(value)

    def _slots(self, ids):
        """ids -> (ids int64, their slots, found): searchsorted in the monotone slot -> id map.  An id outside
        [idx_base, idx_base + max(capacity, ids issued)) raises MdirError; found is False for an id no used slot holds
        (never issued, or purged by compact())."""
        a = check_ids(ids, self.idx_base, self.idx_base + max(self.n, self._next_id)) + self.idx_base
        pos = np.searchsorted(self._ids, a)
        found = pos < self._ids.size
        found[found] = self._ids[pos[found]] == a[found]
        return a, pos, found

    def remove(self, ids):
        """Hide the rows with these ids from every later search.  Stream-ordered on the current stream; removing a
        removed (or purged) id is a no-op; an id outside this index raises MdirError."""
        _, pos, found = self._slots(ids)
        with torch.cuda.device(self.device):
            self._set_live(pos[found], 0)

    def restore(self, ids):
        """Undo remove() for these ids (the rows' data never left the device).  An id that compact() purged, one that
        add() never issued, or one outside this index raises MdirError."""
        a, pos, found = self._slots(ids)
        if not found.all():
            bad = int(a[~found][0])
            if bad < self.idx_base + self._next_id:
                raise _lib.MdirError("id %d was removed and then purged by compact(); it cannot be restored" % bad)
            raise _lib.MdirError("id %d names a slot that was never filled" % bad)
        with torch.cuda.device(self.device):
            self._set_live(pos, 1)

    def add(self, vecs):
        """Append (m, D) fp32 rows to the next free slots; returns their ids (int64 host tensor), which continue from the
        highest id ever issued (idx_base + slot until the first compact()); idx_base + ids issued must stay <= 2**32.
        In stream order: bf16 rows, fp32 master rows, int8 rows + certificate stats (when built), the id map and scan
        extent, then the live bits, so a search queued after this call sees the new rows and one queued before it does
        not.  New rows can only widen the certificate's bounds: the first-pass route chosen earlier stays and stays
        exact.  MdirError when the rows do not fit the capacity."""
        lib = _lib.lib()
        with torch.cuda.device(self.device):
            v = _as_dev_f32(vecs, self.device)
            if v.dim() != 2 or v.shape[1] != self.D:
                raise _lib.MdirError("add() expects (m, %d) rows, got %s" % (self.D, tuple(v.shape)))
            m, s0 = int(v.shape[0]), self._n_used
            if s0 + m > self.n:
                raise _lib.MdirError("index is full: %d free slots, %d rows given" % (self.n - s0, m))
            if m == 0:
                return torch.empty((0,), dtype=torch.int64)
            if self.idx_base + self._next_id + m > 1 << 32:
                raise _lib.MdirError("ids would pass 2**32: %d issued from idx_base %d" % (self._next_id, self.idx_base))
            s1 = s0 + m
            pack_bf16(v, out=self.db16[s0:s1])
            if self.db32 is not None:
                self.db32[s0:s1].copy_(v)
            if self._stats is not None:
                # the stats of the new rows merged into the live ones by max: the same values as one pass over every row
                st = torch.zeros((4,), dtype=torch.float32, device=self.device)
                if self.db8 is not None:
                    _lib.check(lib.mdir_pack_stats_i8(_lib.ptr(self.db32[s0:s1]), _lib.ptr(self.db16[s0:s1]), m, self.D, _lib.ptr(st),
                                                      _lib.ptr(self.db8[s0:s1]), _lib.ptr(self.row_scale[s0:s1]), _lib.stream()),
                               "mdir_pack_stats_i8")
                else:
                    _lib.check(lib.mdir_pack_stats(_lib.ptr(self.db32[s0:s1]), _lib.ptr(self.db16[s0:s1]), m, self.D, _lib.ptr(st),
                                                   _lib.stream()), "mdir_pack_stats")
                torch.maximum(self._stats, st, out=self._stats)
            ids = self._issue_ids(m)
            self.slot_id[s0:s1].copy_(torch.from_numpy(ids.astype(np.uint32).view(np.int32)))
            self.n_scan.fill_(s1)
            self._set_live(np.arange(s0, s1, dtype=np.int64), 1)
            return torch.from_numpy(ids)

    def _issue_ids(self, m):
        """Host bookkeeping of add(): the ids of m rows appended at slot _n_used, continuing from the highest id issued."""
        ids = np.arange(self.idx_base + self._next_id, self.idx_base + self._next_id + m, dtype=np.int64)
        self._ids = np.concatenate([self._ids, ids])
        self._next_id += m
        self._n_used += m
        return ids

    def _compacted_mirrors(self, keep):
        """Host bookkeeping of compact(): the used slots `keep` (ascending) are now slots [0, len(keep))."""
        self._ids = self._ids[keep]
        self._live_host[:] = False
        self._live_host[:keep.size] = True
        self._n_used = int(keep.size)

    def compact(self):
        """Move the live rows to slots [0, n_live), keeping their order, in every plane (bf16 rows, fp32 master, int8
        rows and scales, the slot -> id map); zero the freed slots; shrink the scan extent to n_live.  Removed rows are
        purged: their data is gone from the device, restore() of their ids raises, and add() refills the freed slots with
        new ids.  Ids of live rows do not change.  Returns the number of rows purged (0: nothing launched).  Stream-ordered
        on the current stream; the certificate stats are kept (maxima over a superset of the rows: still a bound).  An Index
        built from a device fp32 tensor with capacity == n keeps that tensor as its master copy, so this rewrites it."""
        used = self._live_host[:self._n_used]
        keep = np.flatnonzero(used)
        purged = self._n_used - keep.size
        if purged == 0:
            return 0
        self._mutations += 1
        lib = _lib.lib()
        sched = compaction_schedule(used, self.compact_chunk)
        with torch.cuda.device(self.device):
            n_words = self.live.numel()
            prefix = torch.empty((n_words + 1,), dtype=torch.int64, device=self.device)
            _lib.check(lib.mdir_compact_prefix(_lib.ptr(self.live), n_words, _lib.ptr(prefix), _lib.stream()), "mdir_compact_prefix")
            staged = max([c[3] for c in sched if c[4]], default=0)
            sbytes = lib.mdir_compact_scratch_bytes(staged, self.D, int(self.db32 is not None), int(self.db8 is not None)) if staged else 0
            scratch = torch.empty((sbytes,), dtype=torch.uint8, device=self.device) if staged else None
            planes = (_lib.ptr(self.db16), _lib.ptr(self.db32), _lib.ptr(self.db8), _lib.ptr(self.row_scale), _lib.ptr(self.slot_id))
            for lo, hi, dst0, n_dst, st in sched:
                _lib.check(lib.mdir_compact_move(*planes, self.n, self.D, _lib.ptr(self.live), _lib.ptr(prefix), lo, hi, dst0, n_dst,
                                                 _lib.ptr(scratch if st else None), sbytes if st else 0, _lib.stream()), "mdir_compact_move")
            _lib.check(lib.mdir_compact_finish(*planes, self.D, _lib.ptr(self.live), n_words, keep.size, self._n_used, _lib.ptr(self.n_scan),
                                               _lib.stream()), "mdir_compact_finish")
        self._compacted_mirrors(keep)
        self._db_x3 = None                         # scores(precision="fp32") split of the old layout
        return int(purged)

    @contextlib.contextmanager
    def _live_version(self, live):
        """Searches inside the block read `live` (an earlier copy of the bitmap) instead of the current one."""
        if live is None:
            yield
            return
        cur, self.live = self.live, live
        try:
            yield
        finally:
            self.live = cur

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
    def _buf(self, name, shape, dtype, ws=None):
        """The device buffer (name, shape, dtype) of workspace ws (a dict; default: the index's own), allocated once."""
        ws = self._ws if ws is None else ws
        key = (name, tuple(shape), dtype)
        b = ws.get(key)
        if b is None:
            b = ws[key] = torch.empty(shape, dtype=dtype, device=self.device)
        return b

    def _route(self, kth, nq):
        """The top-k first pass of a block of nq queries at selection depth kth -> (route, n_sample, stride):
        mdir_topk_plan on the capacity and this device's SM count.  Route 0 = dense, 1 = one-launch (each persistent CTA
        samples one tile; taken while the candidate segments stay at most half full), 2 = sample / select / filter with
        n_sample tiles at that stride (a sample that grows with the database: larger k or databases).  The one-launch
        route is demoted to the three-launch plan (dense when there is none) when `fused` is off or nq > MAX_Q."""
        if self._sms is None:
            self._sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        route, n_sample, stride = topk_plan(self.n, kth, self._sms)
        if route == 1 and (not self.fused or nq > MAX_Q):
            route = 2 if n_sample else 0
        return route, n_sample, stride

    def _fused_ok(self, kth, nq=1):
        """True when a block of nq queries at selection depth kth takes the one-launch route."""
        return self._route(kth, nq)[0] == 1

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

    def _pack_q_i8(self, q32, ws=None):
        """q32 (nq, D) fp32 -> the int8 first pass's query operand (q8 = two int8 planes, their scales) and the per-query
        bounds q_eps of its certificate (mdir_pack_q_i8), in workspace ws."""
        nq = q32.shape[0]
        n_pad = -(-nq // 16) * 16
        q8 = self._buf("q8", (2 * n_pad, self.D), torch.int8, ws)
        qsc = self._buf("q8_scale", (nq, 2), torch.float32, ws)
        qeps = self._buf("q8_eps", (nq,), torch.float32, ws)
        _lib.check(_lib.lib().mdir_pack_q_i8(_lib.ptr(q32), nq, self.D, _lib.ptr(self.stats()), _lib.ptr(q8), _lib.ptr(qsc), _lib.ptr(qeps),
                                             _lib.stream()), "mdir_pack_q_i8")
        return (q8, qsc), qeps

    def _scan(self, q16, mode, stride, n_sample, dense, dense_ld, tau, cand, cnt):
        # more than 128 queries: one WIDE launch, work items = (tile, 128-query block) -- one kernel ramp, and a database
        # tile comes from HBM once for all the blocks (the tensor-bound regime: DBA, all-pairs)
        fn = _lib.lib().mdir_sim_scan_wide_bf16_extent if q16.shape[0] > MAX_Q else _lib.lib().mdir_sim_scan_bf16_extent
        _lib.check(fn(_lib.ptr(self.db16), self.n, _lib.ptr(q16), q16.shape[0], self.D, mode, stride,
                      n_sample, _lib.ptr(dense), dense_ld, _lib.ptr(tau), self.idx_base, _lib.ptr(cand),
                      _lib.ptr(cnt), CAP_S, CAP_L, _lib.ptr(self.live), _lib.ptr(self.n_scan), _lib.stream()), "mdir_sim_scan_bf16_extent")

    def _cand_bufs(self, nq=MAX_Q_WIDE, ws=None):
        rows = MAX_Q_WIDE if nq <= MAX_Q_WIDE else WIDE_Q
        return (self._buf("tau", (rows,), torch.int64, ws), self._buf("cand", (rows, CAND_ROW), torch.int64, ws),
                self._buf("segcnt", (rows, N_SEGS), torch.int32, ws))

    def _first_pass(self, route, q, kth, nq, ws=None):
        """The first pass of the top-kth of one block of nq queries, into the candidate buffers of workspace ws ->
        (tau, cand, cnt, caps) for _finalize.  route = (route, n_sample, stride) of _route; q = the bf16 queries (nq, D),
        or on the one-launch route the int8 operand of _pack_q_i8.
        Dense (route 0): every score -> exact kth-key select; the route for small databases and the recovery after a
        candidate segment overflowed (the select emits exactly kth keys, so nothing can overflow here).  Three-launch
        (route 2): SAMPLE scan -> select the threshold -> FILTER scan; one WIDE launch each beyond MAX_Q queries.
        One-launch (route 1): threshold and filter inside the bf16 or int8 scan.
        self.prof (bench.py: CUDA events on the launch stream) brackets the dominant kernel with its algorithmic bytes."""
        lib = _lib.lib()
        r, n_sample, stride = route
        tau, cand, cnt = self._cand_bufs(nq, ws)     # the select / fused kernel (re)initialises every segment counter
        prof = getattr(self, "prof", None)
        if r == 1:
            rest = (kth, _lib.ptr(tau), self.idx_base, _lib.ptr(cand), _lib.ptr(cnt), 0, FUSED_CAP_L, _lib.ptr(self._fused_ws()),
                    _lib.ptr(self.live), _lib.ptr(self.n_scan), _lib.stream())
            if prof is not None:
                prof.begin()
            if isinstance(q, tuple):
                _lib.check(lib.mdir_sim_scan_fused_i8_extent(_lib.ptr(self.db8), _lib.ptr(self.row_scale), self.n, _lib.ptr(q[0]), _lib.ptr(q[1]),
                                                             nq, self.D, *rest), "mdir_sim_scan_fused_i8_extent")
                nbytes = self.n * self.D + 4 * self.n       # int8 rows + their fp32 scales
            else:
                _lib.check(lib.mdir_sim_scan_fused_bf16_extent(_lib.ptr(self.db16), self.n, _lib.ptr(q), nq, self.D, *rest),
                           "mdir_sim_scan_fused_bf16_extent")
                nbytes = self.n * self.D * 2
            if prof is not None:
                prof.end(nbytes)
            return tau, cand, cnt, (0, FUSED_CAP_L)
        # scores of every row (dense) or of the sampled tiles (SAMPLE mode 1) -> the select kernel
        sampled = int(r == 2)
        if not sampled:
            rows = ld = self.n
            scores = self._buf("dense", (MAX_Q if nq <= MAX_Q else (MAX_Q_WIDE if nq <= MAX_Q_WIDE else WIDE_Q), max(self.n, 1)), torch.float32, ws)
        elif nq <= MAX_Q_WIDE:
            rows, ld = n_sample * TILE, MAX_SAMPLE_TILES * TILE
            scores = self._buf("sample", (MAX_Q if nq <= MAX_Q else MAX_Q_WIDE, ld), torch.float32, ws)
        else:
            rows = ld = n_sample * TILE
            scores = self._buf("sample_wide", (WIDE_Q, rows), torch.float32, ws)
        self._scan(q, sampled, stride, n_sample, scores, ld, None, None, None)
        _lib.check(lib.mdir_select_kth_live(_lib.ptr(scores), ld, rows, nq, kth, stride, self.idx_base, _lib.ptr(tau), _lib.ptr(cand),
                                            CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, sampled, _lib.ptr(self.live), _lib.stream()), "mdir_select_kth_live")
        if sampled:
            if prof is not None:
                prof.begin()
            self._scan(q, 2, stride, n_sample, None, 0, tau, cand, cnt)
            if prof is not None:
                prof.end((self.n - rows) * self.D * 2)
        return tau, cand, cnt, (CAP_S, CAP_L)

    def _finalize(self, cand, cnt, nq, kth, out_scores, out_idx, out_keys, tau, ovf, rescore=None, caps=(CAP_S, CAP_L), q_eps=None):
        """rescore = (q32_block, k_out): fused exact fp32 re-scoring of the kth-long bf16 shortlist.
        q_eps: per-query bounds of the int8 first pass (certified, instead of the bf16 bound); with `tiered` its
        extension is re-scored from the bf16 rows first and only the rows inside their bound from fp32."""
        CAP_S, CAP_L = caps
        CAND_ROW = CAP_S + 148 * CAP_L            # the row stride the scan kernels derive from the two capacities
        if rescore is None:
            _lib.check(_lib.lib().mdir_topk_finalize_ids(_lib.ptr(cand), CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, CAP_L, nq, kth,
                                                         _lib.ptr(out_scores), _lib.ptr(out_idx), _lib.ptr(out_keys), _lib.ptr(tau),
                                                         _lib.ptr(ovf), self.idx_base, _lib.ptr(self.slot_id), _lib.stream()), "mdir_topk_finalize_ids")
        elif q_eps is not None and self.tiered:
            q32, k_out = rescore
            _lib.check(_lib.lib().mdir_topk_finalize_rescore_tiered_ids(_lib.ptr(cand), CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, CAP_L, nq, kth,
                                                                        k_out, _lib.ptr(self.db32), _lib.ptr(self.db16), self.n, self.idx_base,
                                                                        _lib.ptr(q32), self.D, _lib.ptr(self.stats()), _lib.ptr(q_eps),
                                                                        _lib.ptr(out_scores), _lib.ptr(out_idx), _lib.ptr(out_keys), _lib.ptr(tau),
                                                                        _lib.ptr(ovf), _lib.ptr(self.slot_id), _lib.stream()),
                       "mdir_topk_finalize_rescore_tiered_ids")
        elif q_eps is not None:
            q32, k_out = rescore
            _lib.check(_lib.lib().mdir_topk_finalize_rescore_eps_ids(_lib.ptr(cand), CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, CAP_L, nq, kth, k_out,
                                                                     _lib.ptr(self.db32), self.n, self.idx_base, _lib.ptr(q32), self.D,
                                                                     _lib.ptr(self.stats()), _lib.ptr(q_eps), _lib.ptr(out_scores),
                                                                     _lib.ptr(out_idx), _lib.ptr(out_keys), _lib.ptr(tau), _lib.ptr(ovf),
                                                                     _lib.ptr(self.slot_id), _lib.stream()), "mdir_topk_finalize_rescore_eps_ids")
        else:
            q32, k_out = rescore
            stats = self.stats() if self.certify else None
            _lib.check(_lib.lib().mdir_topk_finalize_rescore_ids(_lib.ptr(cand), CAND_ROW, _lib.ptr(cnt), N_SEGS, CAP_S, CAP_L, nq, kth, k_out,
                                                                 _lib.ptr(self.db32), self.n, self.idx_base, _lib.ptr(q32), self.D,
                                                                 _lib.ptr(stats), _lib.ptr(out_scores), _lib.ptr(out_idx), _lib.ptr(out_keys),
                                                                 _lib.ptr(tau), _lib.ptr(ovf), _lib.ptr(self.slot_id), _lib.stream()),
                       "mdir_topk_finalize_rescore_ids")

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
        """The top-kth of one block: the first pass _route chooses, then _finalize.  q16 None: the int8 first pass
        (Index._i8_route); a block it flags (bit 0 or 1) is redone here through the bf16 route when check=True -- the
        int8 pass never widens, recovery is the bf16 route's own."""
        nq = ovf.shape[0]

        def topk(route, q, kth, q_eps=None):
            tau, cand, cnt, caps = self._first_pass(route, q, kth, nq)
            self._finalize(cand, cnt, nq, kth, out_s, out_i, out_k, tau, ovf, rescore, caps, q_eps)

        if q16 is None:
            self.route = "int8"
            self.cert["int8_blocks"] += 1
            q8, q_eps = self._pack_q_i8(rescore[0])
            topk(self._route(kth, nq), q8, kth, q_eps)
            if not check:
                return
            st = ovf.cpu()
            if not bool(st.any()):
                self.cert["queries"] += int(st.numel())
                return
            self.cert["int8_redone"] += 1
            q16 = pack_bf16(rescore[0])
        self.route = "bf16"
        topk(self._route(kth, nq), q16, kth)
        if not check:
            return
        st = ovf.cpu()
        self.cert["queries"] += int(st.numel())
        if bool((st & STATUS_OVERFLOW).any()):
            # a candidate segment overflowed (adversarial row order / massive ties): exact dense route
            topk(DENSE_ROUTE, q16, kth)
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
            topk(self._route(kth, nq), q16, kth)
            st = ovf.cpu()
            if bool((st & STATUS_OVERFLOW).any()):
                topk(DENSE_ROUTE, q16, kth)
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

    def range_search(self, q, min_score, precision="fp32", check=True):
        """Every live row whose score against query i is >= min_score (a float, or a (N_q,) tensor: one per query).
        q: (N_q, D) fp32 (host or device).  Returns (lims (N_q + 1,) int64, scores fp32, ids int32), all on the device, in
        the CSR layout of FAISS range_search: the results of query i are scores / ids[lims[i]:lims[i + 1]], ordered by
        (score desc, id asc) as search() orders them; ids go through the slot -> id map.

        precision="fp32": the exact fp32 score, in the one summation order search(precision="fp32") uses for every
                          row, so a row's range score is its search score bit for bit.  The bf16 scan
                          passes every row within the certified bound eps of min_score; those rows are re-scored in fp32
                          and filtered, so the result is complete by construction (no threshold to guess, no widening).
        precision="bf16": the bf16-input / fp32-accumulate scan score, as search(precision="bf16") reports it.
        One scan per block of 128 queries.  A candidate segment that overflowed is visible in the scan's exact counts;
        check=True re-scans that block once with segments sized from them (in smaller query groups when they exceed
        RANGE_BUDGET; range_stats counts both), check=False returns the block as it is with status bit 0 raised for the
        truncated queries (status() / check_overflow()).  NaN in min_score raises MdirError."""
        lib = _lib.lib()
        with torch.cuda.device(self.device):
            q32 = _as_dev_f32(q, self.device)
            if q32.dim() != 2 or q32.shape[1] != self.D:
                raise _lib.MdirError("range_search expects (N_q, %d) queries, got %s" % (self.D, tuple(q32.shape)))
            if precision == "fp32":
                if self.db32 is None:
                    raise _lib.MdirError("precision='fp32' needs keep_fp32=True")
            elif precision != "bf16":
                raise ValueError("precision must be 'fp32' or 'bf16'")
            nq_all = q32.shape[0]
            m_host = range_thresholds(min_score, nq_all)
            parts = []                          # (counts, scores, ids, status) of consecutive query groups
            if nq_all and self._n_used:       # an index with every row removed scans and returns nothing
                m_all = torch.from_numpy(m_host).to(self.device)
                stats = self.stats() if precision == "fp32" else None
                q16 = pack_bf16(q32)
                tau = torch.empty((nq_all,), dtype=torch.int64, device=self.device)
                _lib.check(lib.mdir_range_tau(_lib.ptr(q32), nq_all, self.D, _lib.ptr(m_all), _lib.ptr(stats), _lib.ptr(tau), _lib.stream()),
                           "mdir_range_tau")
                for q0 in range(0, nq_all, MAX_Q):
                    q1 = min(q0 + MAX_Q, nq_all)
                    parts += self._range_block(q16[q0:q1], q32[q0:q1], m_all[q0:q1], tau[q0:q1], stats, check)
                self.range_stats["queries"] += nq_all
            else:
                parts.append((np.zeros((nq_all,), dtype=np.int64), torch.empty((0,), dtype=torch.float32, device=self.device),
                              torch.empty((0,), dtype=torch.int32, device=self.device), np.zeros((nq_all,), dtype=np.int32), None))
            status = np.concatenate([p[3] for p in parts])
            self._ovf = torch.from_numpy(status).to(self.device) if status.any() else torch.zeros((nq_all,), dtype=torch.int32, device=self.device)
            if len(parts) == 1:
                out_s, out_i, lims = parts[0][1], parts[0][2], parts[0][4]
            else:
                out_s, out_i, lims = torch.cat([p[1] for p in parts]), torch.cat([p[2] for p in parts]), None
            if lims is None:                    # several groups (or nothing to emit): offsets of the concatenation
                lims_h = np.zeros((nq_all + 1,), dtype=np.int64)
                np.cumsum(np.concatenate([p[0] for p in parts]), out=lims_h[1:])
                lims = torch.from_numpy(lims_h).to(self.device)
            return lims, out_s, out_i

    def _range_block(self, q16, q32, m, tau, stats, check):
        """One block of <= 128 queries -> [(counts, scores, ids, status, lims)] for consecutive groups of its queries."""
        nq = q16.shape[0]
        self.range_stats["blocks"] += 1
        bufs = self._range_bufs(RANGE_CAP_L, MAX_Q)
        run_len, max_seg = self._range_pass(q16, q32, m, tau, stats, RANGE_CAP_L, bufs)
        over = max_seg > RANGE_CAP_L
        if not check or not over.any():
            return [self._range_emit(bufs, run_len, over)]
        # the exact counts say how deep every segment has to be: one re-scan, in query groups that fit the budget
        self.range_stats["rescans"] += 1
        cap, group = range_rescan_plan(max_seg)
        out = []
        for g0 in range(0, nq, group):
            g1 = min(g0 + group, nq)
            self.range_stats["rescan_groups"] += 1
            bufs = self._range_bufs(cap, g1 - g0, {})         # a workspace of its own: freed with the call
            run_len, max_seg = self._range_pass(q16[g0:g1], q32[g0:g1], m[g0:g1], tau[g0:g1], stats, cap, bufs)
            if (max_seg > cap).any():
                raise _lib.MdirError("range_search re-scan overflowed its exact capacity (internal error)")
            out.append(self._range_emit(bufs, run_len, max_seg > cap))
        return out

    def _range_bufs(self, cap_l, rows, ws=None):
        """Candidate rows, segment counts, survivors and the gather's per-chunk counts + max segment counts of a range
        scan with segment capacity cap_l, from workspace ws (default: the index's own, under names apart from search()'s
        candidate buffers, so a range call never changes a later search)."""
        n_chunks = range_chunks(cap_l)
        return (self._buf("range_cand", (rows, 148 * cap_l), torch.int64, ws), self._buf("range_segcnt", (rows, N_SEGS), torch.int32, ws),
                self._buf("range_surv", (rows, n_chunks * RANGE_CHUNK), torch.int64, ws),
                self._buf("range_runs", (rows * (n_chunks + 1),), torch.int32, ws))

    def _range_pass(self, q16, q32, m, tau, stats, cap_l, bufs):
        """_range_launch, then run_len (nq, n_chunks) and max_seg (nq,) read back in one copy (the call's synchronisation
        point)."""
        nq = q16.shape[0]
        n_chunks = range_chunks(cap_l)
        self._range_launch(q16, q32, m, tau, stats, cap_l, bufs)
        host = bufs[3][:nq * (n_chunks + 1)].cpu().numpy()
        return host[:nq * n_chunks].reshape(nq, n_chunks), host[nq * n_chunks:]

    def _range_launch(self, q16, q32, m, tau, stats, cap_l, bufs):
        """FILTER scan of every used slot at threshold tau, then the gather -> device views (run_len (nq * n_chunks,),
        max_seg (nq,)) of bufs' runs.  No host synchronisation (GraphedRangeSearch captures it).  stats None: bf16
        scores, no re-scoring."""
        lib = _lib.lib()
        nq = q16.shape[0]
        cand, cnt, surv, runs = bufs
        n_chunks = range_chunks(cap_l)
        cnt[:nq].zero_()                    # the scan writes the segments of the CTAs it launches; the rest stay empty
        prof = getattr(self, "prof", None)
        if prof is not None:
            prof.begin()
        _lib.check(lib.mdir_sim_scan_bf16_extent(_lib.ptr(self.db16), self.n, _lib.ptr(q16), nq, self.D, 2, 0, 0, None, 0, _lib.ptr(tau),
                                                 self.idx_base, _lib.ptr(cand), _lib.ptr(cnt), 0, cap_l, _lib.ptr(self.live),
                                                 _lib.ptr(self.n_scan), _lib.stream()), "mdir_sim_scan_bf16_extent")
        if prof is not None:
            prof.end(self._n_used * self.D * 2)
        run_len, max_seg = runs[:nq * n_chunks], runs[nq * n_chunks:nq * (n_chunks + 1)]
        _lib.check(lib.mdir_range_gather(_lib.ptr(cand), 148 * cap_l, _lib.ptr(cnt), cap_l, nq, _lib.ptr(m),
                                         _lib.ptr(self.db32 if stats is not None else None), self.n, self.idx_base, _lib.ptr(q32), self.D,
                                         _lib.ptr(surv), n_chunks, _lib.ptr(run_len), _lib.ptr(max_seg), _lib.stream()), "mdir_range_gather")
        return run_len, max_seg

    def _range_emit(self, bufs, run_len, over):
        """Sorted CSR output of one range pass -> (counts, scores, ids, status, lims on the device or None) of its queries."""
        lib = _lib.lib()
        _, _, surv, runs = bufs
        nq, n_chunks = run_len.shape
        counts, lims, run_off = range_csr(run_len)
        total = int(lims[-1])
        scores = torch.empty((total,), dtype=torch.float32, device=self.device)
        ids = torch.empty((total,), dtype=torch.int32, device=self.device)
        lims_d = None
        if total:
            lims_d = torch.from_numpy(lims).to(self.device)
            small = counts[(counts > 0) & (counts <= RANGE_STAGE)]
            if small.size:
                stage = 32
                while stage < int(small.max()):
                    stage *= 2
                off_d = torch.from_numpy(run_off).to(self.device)
                _lib.check(lib.mdir_range_emit(_lib.ptr(surv), n_chunks, _lib.ptr(runs), _lib.ptr(off_d), _lib.ptr(lims_d), nq, stage, self.idx_base,
                                               _lib.ptr(self.slot_id), _lib.ptr(scores), _lib.ptr(ids), _lib.stream()), "mdir_range_emit")
            big = np.flatnonzero(counts > RANGE_STAGE).astype(np.int32)
            if big.size:
                self.range_stats["large_sorts"] += int(big.size)
                rows = torch.from_numpy(big).to(self.device)
                _lib.check(lib.mdir_range_sort_runs(_lib.ptr(surv), n_chunks, _lib.ptr(runs), _lib.ptr(rows), int(big.size), _lib.stream()),
                           "mdir_range_sort_runs")
                _lib.check(lib.mdir_range_merge(_lib.ptr(surv), n_chunks, _lib.ptr(runs), _lib.ptr(rows), int(big.size), _lib.ptr(lims_d),
                                                self.idx_base, _lib.ptr(self.slot_id), _lib.ptr(scores), _lib.ptr(ids), _lib.stream()),
                           "mdir_range_merge")
        status = np.where(np.asarray(over, dtype=bool), STATUS_OVERFLOW, 0).astype(np.int32)
        return counts, scores, ids, status, lims_d

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
        tf32 / fp32 need the fp32 master copy (keep_fp32=True); fp32 caches a 3x-wide split of it.
        Every slot is scored, so an index with removed rows or free capacity raises MdirError."""
        self._require_all_live("Index.scores()")
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
        max_pairs // N_db to bound the sort workspace (~30 B per pair).  An index with removed rows or free capacity
        raises MdirError."""
        self._require_all_live("Index.ranks()")
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

    def _id_ranges(self):
        """(first id, end id) of every rank's shard, gathered once: a collective, like remove() / restore()."""
        if getattr(self, "_ranges", None) is None:
            loc = self.local
            if self.world == 1:
                self._ranges = [(loc.idx_base, loc.idx_base + loc.n)]
            else:
                dev = self.device if self.dist.get_backend(self.group) == "nccl" else torch.device("cpu")
                mine = torch.tensor([loc.idx_base, loc.idx_base + loc.n], dtype=torch.int64, device=dev)
                allr = torch.empty((self.world * 2,), dtype=torch.int64, device=dev)
                self.dist.all_gather_into_tensor(allr, mine, group=self.group)
                r = allr.cpu().tolist()
                self._ranges = [(int(r[2 * i]), int(r[2 * i + 1])) for i in range(self.world)]
        return self._ranges

    def _local_ids(self, ids):
        rank = self.dist.get_rank(self.group) if self.world > 1 else 0
        return ids_for_rank(ids, self._id_ranges(), rank)

    def remove(self, ids):
        """Index.remove with GLOBAL ids: every rank makes the same call with the same list and applies the ids its shard
        owns.  An id in no rank's shard raises MdirError (on every rank)."""
        self.local.remove(self._local_ids(ids))

    def restore(self, ids):
        """Index.restore with GLOBAL ids, called by every rank with the same list (see remove())."""
        self.local.restore(self._local_ids(ids))

    def compact(self):
        """Index.compact of this rank's shard, called by every rank at the same point of its sequence (like remove()).
        The ids and every rank's id range are unchanged.  Returns the rows this shard purged."""
        return self.local.compact()

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
        # the graphs' own candidate, status and query buffers: eager searches between replays leave them alone (the fused
        # scan's arrival counters are shared: zeroed once, re-armed by the kernel itself)
        self._ws = ws = {}
        route = loc._route(self.kth, nq)
        i8 = loc._i8_route(self.kth, nq)         # the same route choice as Index.search
        self.keys = torch.empty((nq, k), dtype=torch.int64, device=dev)
        self.local_out = (torch.empty((nq, k), dtype=torch.float32, device=dev), torch.empty((nq, k), dtype=torch.int32, device=dev))
        self.ovf = loc._buf("ovf", (max(nq, 1),), torch.int32, ws)[:nq]
        if self._has_exchange:
            self.out = (torch.empty((nq, k), dtype=torch.float32, device=dev), torch.empty((nq, k), dtype=torch.int32, device=dev))
            self.status = torch.zeros((nq,), dtype=torch.int32, device=dev)
        else:
            self.out, self.status = self.local_out, self.ovf

        def front():
            q_eps = None
            if i8:
                q, q_eps = loc._pack_q_i8(self.q, ws)
            else:
                q = pack_bf16(self.q, out=loc._buf("q16", (nq, loc.D), torch.bfloat16, ws))
            lib.mdir_tune(1, self.scan_ctas)
            try:
                return loc._first_pass(route, q, self.kth, nq, ws), q_eps
            finally:
                lib.mdir_tune(1, 0)

        def back(first):
            (tau, cand, cnt, caps), q_eps = first
            chunk = self.fin_chunk if self.fin_chunk > 0 else nq
            lib.mdir_tune(2, 0 if self.fin_chunk > 0 else 1)
            lib.mdir_tune(3, self.fin_stage)
            try:
                for q0 in range(0, nq, chunk):
                    q1 = min(q0 + chunk, nq)
                    loc._finalize(cand[q0:q1], cnt[q0:q1], q1 - q0, self.kth, self.local_out[0][q0:q1], self.local_out[1][q0:q1],
                                  self.keys[q0:q1], tau[q0:q1], self.ovf[q0:q1], (self.q[q0:q1], k), caps=caps,
                                  q_eps=None if q_eps is None else q_eps[q0:q1])
            finally:
                lib.mdir_tune(2, 1)
                lib.mdir_tune(3, 0)
            if self._has_exchange:
                # the NVLink push + merge of these keys rides in the same graph: one launch per ticket on the side stream
                self.index._exchange(self.keys, nq, k, 0, self.out[0], self.out[1], self.ovf, self.status)

        with torch.cuda.device(dev):
            loc.prof = prof                      # the scan's event pair: recorded in the warm-up too, captured in `graph`
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(2):
                    back(front())
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            self.graph, self.back = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                first = front()
            with torch.cuda.graph(self.back):
                back(first)
            loc.prof = None
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


class _Pipeline:
    """The ticket slots and the mutation ordering that SearchPipeline and RangePipeline share.  A subclass sets index,
    local, depth, overlap, the streams compute / d2h (and exch when overlap) and self.slots: one dict per slot with at
    least "pending" (a ticket is in flight) and "live" (the bitmap copy its recovery reads, None: the current one)."""

    def _mutate(self, fn):
        """Run a mutation of the index on the compute stream, after every replay already queued there (and, in overlap
        mode, after the finalize / exchange queued on the exchange stream, which read the rows and stats that add()
        writes).  Tickets in flight keep a device copy of the live bitmap they were submitted with: a ticket redone by
        result()'s recovery path then sees the same rows as its replay did.  A copy is dropped when its last ticket is
        collected."""
        dev = self.local.device
        with torch.cuda.device(dev):
            if self.overlap:
                self.compute.wait_stream(self.exch)
            with torch.cuda.stream(self.compute):
                waiting = [sl for sl in self.slots if sl["pending"] and sl["live"] is None]
                if waiting:
                    snap = self.local.live.clone()
                    for sl in waiting:
                        sl["live"] = snap
                return fn()

    def remove(self, ids):
        """index.remove(ids) between tickets: tickets submitted before this call do not see it, later ones do.  With a
        ShardedIndex, ids are global and every rank makes the same call at the same point of its ticket sequence."""
        self._mutate(lambda: self.index.remove(ids))

    def restore(self, ids):
        """index.restore(ids) between tickets (see remove())."""
        self._mutate(lambda: self.index.restore(ids))

    def add(self, vecs):
        """index.add(vecs) between tickets (see remove()); returns the new ids.  Single-GPU Index only."""
        if isinstance(self.index, ShardedIndex):
            raise _lib.MdirError("%s.add() needs an Index: ShardedIndex has no add()" % type(self).__name__)
        return self._mutate(lambda: self.index.add(vecs))

    def compact(self):
        """index.compact() on the compute stream, after the replays and exchanges already queued.  A maintenance step:
        collect every ticket first -- MdirError while one is pending, because the live-row copy a ticket keeps for its
        recovery path describes the slot layout compaction changes.  The graphs keep working without re-capture, and
        tickets submitted afterwards see the compacted index.  With a ShardedIndex every rank calls it at the same point.
        Returns the rows purged (on this rank)."""
        pending = [sl for sl in self.slots if sl["pending"]]
        if pending:
            raise _lib.MdirError("%s.compact(): collect the %d pending ticket(s) first" % (type(self).__name__, len(pending)))
        return self._mutate(self.index.compact)

    def _free_slot(self, ticket):
        """The slot of a ticket about to be submitted; MdirError while the ticket `depth` before it is uncollected."""
        slot = self.slots[ticket % self.depth]
        if slot["pending"]:
            raise _lib.MdirError("%s: collect result() of ticket %d before submitting more" % (type(self).__name__, ticket - self.depth))
        return slot

    def _pending_slot(self, ticket):
        """The slot of a ticket in flight whose result has not been collected; MdirError otherwise."""
        if not (self.n_submitted - self.depth <= ticket < self.n_submitted):
            raise _lib.MdirError("%s: ticket %d is not in flight" % (type(self).__name__, ticket))
        slot = self.slots[ticket % self.depth]
        if not slot["pending"]:
            raise _lib.MdirError("%s: result(%d) was already collected" % (type(self).__name__, ticket))
        return slot

    def _map(self, batches, submit):
        """Generator of result()s over `batches`, each passed to submit, keeping `depth` tickets in flight."""
        tickets = []
        for b in batches:
            if len(tickets) == self.depth:
                yield self.result(tickets.pop(0))
            tickets.append(submit(b))
        for t in tickets:
            yield self.result(t)


class SearchPipeline(_Pipeline):
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
    With a ShardedIndex every rank must submit the same sequence (the all-gather is inside the graphs).
    remove() / restore() / add() / compact() mutate the index between tickets without re-capturing the graphs."""

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
                    "q": None, "pending": False, "merged": False, "used": False, "live": None})
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
        slot, gs = self._free_slot(t_new), self.graphs[t_new % self.depth]
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
        slot = self._pending_slot(ticket)
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
            # with the live rows this ticket was submitted with (a mutation may have been queued since)
            with torch.cuda.stream(self.compute), self.local._live_version(slot["live"]):
                if sharded:
                    s, i = self.index.search_collective_recovery(slot["q"], self.k, precision=self.precision, shortlist=self.shortlist)
                else:
                    s, i = self.index.search(slot["q"], self.k, precision=self.precision, shortlist=self.shortlist)
                slot["scores"].copy_(s)
                slot["idx"].copy_(i)
            self.compute.synchronize()
        slot["q"], slot["live"] = None, None
        return slot["scores"].numpy(), slot["idx"].numpy()

    def map(self, batches):
        """Generator over an iterable of query batches, keeping `depth` steps in flight."""
        return self._map(batches, self.submit)


class GraphedRangeSearch:
    """One range step (Index.range_search) captured in a CUDA graph: static queries (n_q, D) fp32 and thresholds
    min_score (n_q,) fp32 in, a CSR of static size out -- lims (n_q + 1,) int64, scores / ids arenas of
    n_q * max_results entries (query i at [lims[i], lims[i + 1])) and status (n_q,) int32.

        gr = GraphedRangeSearch(index, n_q=70, max_results=1024)
        lims, scores, ids = gr(q, min_score)      # min_score: a float or one value per query
        gr.check_overflow()                        # after a sync: True -> redo the flagged queries with range_search

    The chain (pack, threshold keys, FILTER scan at RANGE_CAP_L, gather, device CSR offsets, emit) runs without a host
    synchronisation, so the step has no variable-size output.  A query is emitted when its survivors fit max_results
    and no candidate segment overflowed; any other query gets no rows and a status word: STATUS_OVERFLOW (a segment
    overflowed: the graph has no re-scan) and/or STATUS_RANGE_FULL (more than max_results matches).  Whoever owns the
    graph redoes those queries eagerly (RangePipeline does).  Emitted queries are bit for bit those of range_search.
    The graph works in a workspace of its own, so eager calls between replays and replays leave each other unchanged;
    it reads the live bitmap, the scan extent, the slot -> id map and the certificate stats from device memory, so
    remove / restore / add / compact need no re-capture."""

    def __init__(self, index, n_q, max_results=1024, precision="fp32"):
        if isinstance(index, ShardedIndex):
            raise _lib.MdirError("GraphedRangeSearch needs an Index: ShardedIndex has no range_search")
        self.n_q, self.max_results, self.precision = int(n_q), int(max_results), precision
        if not 1 <= self.n_q <= MAX_Q:
            raise _lib.MdirError("GraphedRangeSearch: n_q must be in [1, %d] (got %d)" % (MAX_Q, self.n_q))
        if not 1 <= self.max_results <= RANGE_STAGE:
            raise _lib.MdirError("GraphedRangeSearch: max_results must be in [1, %d] (got %d)" % (RANGE_STAGE, self.max_results))
        if precision == "fp32":
            if index.db32 is None:
                raise _lib.MdirError("precision='fp32' needs keep_fp32=True")
        elif precision != "bf16":
            raise ValueError("precision must be 'fp32' or 'bf16'")
        self.index = loc = index
        dev, nq, D = loc.device, self.n_q, loc.D
        lib = _lib.lib()
        n_chunks = range_chunks(RANGE_CAP_L)
        stage = range_stage_cap(self.max_results)
        with torch.cuda.device(dev):
            stats = loc.stats() if precision == "fp32" else None     # its one read-back happens here, never in the graph
            self.q = torch.zeros((nq, D), dtype=torch.float32, device=dev)
            self.min_score = torch.full((nq,), float("inf"), dtype=torch.float32, device=dev)
            self.lims = torch.zeros((nq + 1,), dtype=torch.int64, device=dev)
            self.scores = torch.empty((nq * self.max_results,), dtype=torch.float32, device=dev)
            self.ids = torch.empty((nq * self.max_results,), dtype=torch.int32, device=dev)
            self.status = torch.zeros((nq,), dtype=torch.int32, device=dev)
            # the graph's other buffers: held by this object (a tensor only the capture used would be freed and its
            # memory handed to later allocations while the graph still writes it)
            self._q16 = q16 = torch.empty((nq, D), dtype=torch.bfloat16, device=dev)
            self._tau = tau = torch.empty((nq,), dtype=torch.int64, device=dev)
            self._run_off = run_off = torch.empty((nq, n_chunks), dtype=torch.int32, device=dev)
            self._ws = {}
            self._bufs = bufs = loc._range_bufs(RANGE_CAP_L, nq, self._ws)
            runs = bufs[3]

            def step():
                _lib.check(lib.mdir_pack_bf16(_lib.ptr(self.q), nq, D, 0, _lib.ptr(q16), _lib.stream()), "mdir_pack_bf16")
                _lib.check(lib.mdir_range_tau(_lib.ptr(self.q), nq, D, _lib.ptr(self.min_score), _lib.ptr(stats), _lib.ptr(tau), _lib.stream()),
                           "mdir_range_tau")
                run_len, max_seg = loc._range_launch(q16, self.q, self.min_score, tau, stats, RANGE_CAP_L, bufs)
                _lib.check(lib.mdir_range_offsets(_lib.ptr(run_len), _lib.ptr(max_seg), nq, n_chunks, RANGE_CAP_L, self.max_results,
                                                  _lib.ptr(self.lims), _lib.ptr(run_off), _lib.ptr(self.status), _lib.stream()),
                           "mdir_range_offsets")
                _lib.check(lib.mdir_range_emit(_lib.ptr(bufs[2]), n_chunks, _lib.ptr(runs), _lib.ptr(run_off), _lib.ptr(self.lims), nq, stage,
                                               loc.idx_base, _lib.ptr(loc.slot_id), _lib.ptr(self.scores), _lib.ptr(self.ids), _lib.stream()),
                           "mdir_range_emit")

            prof, loc.prof = getattr(loc, "prof", None), None            # no timing events inside the graph
            try:
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):                             # warm-up: per-device kernel attributes
                    step()
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    step()
            finally:
                loc.prof = prof

    def __call__(self, q=None, min_score=None):
        """Replay on the current stream.  q: (n_q, D) fp32 (host, pinned for an asynchronous copy, or device) copied into
        the static input; min_score: a float or one value per query (range_thresholds).  None keeps the previous value.
        Returns the static (lims, scores, ids): the result is scores / ids[:lims[n_q]]."""
        if q is not None:
            self.q.copy_(q, non_blocking=True)
        if min_score is not None:
            self.min_score.copy_(torch.from_numpy(range_thresholds(min_score, self.n_q)))
        self.graph.replay()
        return self.lims, self.scores, self.ids

    def check_overflow(self):
        """True when some query of the last replay was flagged (STATUS_OVERFLOW / STATUS_RANGE_FULL) and has no rows:
        redo those queries through index.range_search()."""
        return bool(self.status.any().item())


class RangePipeline(_Pipeline):
    """Host-facing range serving: query batches and thresholds go up from pinned host buffers, GraphedRangeSearch
    replays back to back on one compute stream, and each ticket's CSR comes back in pinned buffers of static size (the
    whole max_results arena per query), copies and replays ordered by events only.

        pipe = RangePipeline(index, n_q=70, max_results=1024)
        t0 = pipe.submit(q_0, 0.4)                 # min_score: a float or one value per query
        t1 = pipe.submit(q_1, m_1)
        lims, scores, ids = pipe.result(t0)        # numpy: query i at [lims[i], lims[i + 1])

    result() is the complete exact answer of range_search(check=True) for every query: a query the graph flagged (a
    candidate segment overflowed, or more than max_results matches) is redone eagerly, with the live rows its ticket
    was submitted with, and spliced into the ticket's CSR (range_splice).  remove() / restore() / add() / compact()
    mutate the index between tickets without re-capturing the graphs."""

    def __init__(self, index, n_q, max_results=1024, depth=2, precision="fp32"):
        if isinstance(index, ShardedIndex):
            raise _lib.MdirError("RangePipeline needs an Index: ShardedIndex has no range_search")
        if int(depth) < 1:
            raise _lib.MdirError("RangePipeline: depth must be at least 1 (got %d)" % int(depth))
        self.graphs = [GraphedRangeSearch(index, n_q, max_results=max_results, precision=precision) for _ in range(int(depth))]
        self.index = self.local = index
        self.n_q, self.max_results, self.precision = int(n_q), int(max_results), precision
        self.depth, self.overlap = int(depth), False
        dev = index.device
        arena = self.n_q * self.max_results
        with torch.cuda.device(dev):
            self.compute, self.h2d, self.d2h = (torch.cuda.Stream(device=dev) for _ in range(3))
            self.slots = [{
                "q": torch.empty((self.n_q, index.D), dtype=torch.float32).pin_memory(),
                "m": torch.empty((self.n_q,), dtype=torch.float32).pin_memory(),
                "lims": torch.empty((self.n_q + 1,), dtype=torch.int64).pin_memory(),
                "status": torch.empty((self.n_q,), dtype=torch.int32).pin_memory(),
                "scores": torch.empty((arena,), dtype=torch.float32).pin_memory(),
                "ids": torch.empty((arena,), dtype=torch.int32).pin_memory(),
                "up": torch.cuda.Event(), "done": torch.cuda.Event(), "down": torch.cuda.Event(),
                "pending": False, "live": None} for _ in range(self.depth)]
            torch.cuda.synchronize(dev)
        self.n_submitted = 0
        self.n_recovered = 0            # tickets with at least one query redone eagerly
        self.recovered = {"overflow": 0, "range_full": 0}     # queries redone, by status bit (a query may count in both)

    def submit(self, q, min_score):
        """q: (n_q, D) fp32 (host or device), min_score: a float or one value per query.  Both are copied into the
        slot's pinned staging buffers here, so the caller may reuse them at once.  Returns a ticket for result()."""
        t_new = self.n_submitted
        slot, gr = self._free_slot(t_new), self.graphs[t_new % self.depth]
        q = torch.as_tensor(q)
        if tuple(q.shape) != tuple(gr.q.shape):
            raise _lib.MdirError("RangePipeline expects query batches of shape %s" % (tuple(gr.q.shape),))
        m = range_thresholds(min_score, self.n_q)
        slot["q"].copy_(q)
        slot["m"].copy_(torch.from_numpy(m))
        with torch.cuda.device(self.local.device):
            with torch.cuda.stream(self.h2d):              # this slot's previous replay was collected by result()
                gr.q.copy_(slot["q"], non_blocking=True)
                gr.min_score.copy_(slot["m"], non_blocking=True)
                slot["up"].record()
            with torch.cuda.stream(self.compute):
                self.compute.wait_event(slot["up"])
                gr.graph.replay()
                slot["done"].record()
            with torch.cuda.stream(self.d2h):
                self.d2h.wait_event(slot["done"])
                for name, src in (("lims", gr.lims), ("status", gr.status), ("scores", gr.scores), ("ids", gr.ids)):
                    slot[name].copy_(src, non_blocking=True)
                slot["down"].record()
        slot["pending"] = True
        self.n_submitted += 1
        return t_new

    def result(self, ticket):
        """Blocks until ticket's CSR is in host memory -> (lims (n_q + 1,) int64, scores fp32, ids int32) numpy.  Views of
        the pinned buffers, valid until `depth` more submits, unless a query was redone: then fresh arrays."""
        slot = self._pending_slot(ticket)
        slot["down"].synchronize()
        slot["pending"] = False
        lims = slot["lims"].numpy()
        n = int(lims[-1])
        out = (lims, slot["scores"].numpy()[:n], slot["ids"].numpy()[:n])
        status = slot["status"].numpy()
        flagged = np.flatnonzero(status)
        if flagged.size:
            self.n_recovered += 1
            self.recovered["overflow"] += int(((status & STATUS_OVERFLOW) != 0).sum())
            self.recovered["range_full"] += int(((status & STATUS_RANGE_FULL) != 0).sum())
            rows = torch.from_numpy(flagged)
            dev = self.local.device
            # on the compute stream (after every replay queued there), with the live rows this ticket was submitted with
            with torch.cuda.device(dev), torch.cuda.stream(self.compute), self.local._live_version(slot["live"]):
                sub = self.index.range_search(slot["q"][rows], slot["m"][rows], precision=self.precision, check=True)
                sub = tuple(t.cpu().numpy() for t in sub)
            out = range_splice(*out, flagged, *sub)
        slot["live"] = None
        return out

    def map(self, batches):
        """Generator over an iterable of (q, min_score) pairs, keeping `depth` tickets in flight."""
        return self._map(batches, lambda b: self.submit(*b))
