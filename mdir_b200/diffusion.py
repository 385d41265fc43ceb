"""Diffusion re-ranking on a mutual kNN graph of the database (Iscen, Tolias, Avrithis, Furon, Chum, CVPR 2017).

NOT in the reference (parity unpinned, like qe.py): the semantics are restated in tests/diffusion_reference.py:diffusion_graph
/ diffusion_search.  The graph is built once per index from the certified fp32 top-(k+1) of every row and kept exact
through add / remove / restore / compact made through the Diffusion (DESIGN 2.2e); a query's
certified fp32 shortlist L is re-ranked by f, the truncated CG solution of (I - alpha S_LL) f = y, where y holds the
query's top k_q scores raised to gamma.  The graph kernels and the per-query solve are mdir_b200/csrc/diffusion.cu.
DiffusionTable is offline diffusion: every row's diffusion solved once, a query combines the rows of its top-k_q
(tests/diffusion_offline_reference.py:offline_table / offline_search).
GraphedDiffusion and DiffusionPipeline serve either one from CUDA graphs (DESIGN 2.2f)."""
import contextlib
import math

import numpy as np
import torch

from . import _lib
from .qe import DBA_BLOCK
from .search import Index, ShardedIndex, MAX_Q, STATUS_OVERFLOW, STATUS_UNCERTIFIED, WIDE_Q, _Pipeline, _as_dev_f32

MAX_K = 255          # neighbours per database row
MAX_TRUNC = 2048     # shortlist rows per query the solve kernel holds in shared memory
MERGE_TILE = 32      # target rows per CTA of mdir_diffusion_merge
MERGE_CAP = 1024     # candidate pairs one tile of the reverse merge holds; a tile with more is re-run with exactly the room it needs
# bytes of the (batch, row chunk) fp32 bf16-score plane of the reverse merge: 1,024 added rows screen 256 Ki rows per
# dense scan, 10,000 rows 26 Ki.  At R1M on a B200 (1,000 W) the 10,000-row scan in 38 chunks ran at ~1,020 TFLOP/s and
# the 1,024-row scan in 4 chunks at ~1,100 (profiles/r12_diffusion_update_1gpu.log); other sizes were not measured.
SCREEN_PLANE_BYTES = 1 << 30
MAX_WIDTH = 1024     # entries per table row of DiffusionTable
MAX_KQ = 128         # table rows one DiffusionTable query combines
MAX_ENTRIES = 8192   # k_q * width (the combine sorts them in shared memory), and the largest k of DiffusionTable.search
# DiffusionTable's build: rows per chunk (one top-trunc search + one mdir_diffusion_solve each) and queries per scan
# pass.  At R1M (width 100, trunc 1000) on a B200 (1,000 W) the search passes took 14.4 s with 128-query passes, 18.1 s
# with 256, 24.1 s with 512 and 31.8 s with 1,024 (WIDE_Q); the solves 0.71 s in chunks of 8,192 rows, 0.80 s in chunks
# of 1,024 and 0.70 s in chunks of 32,768 (profiles/r13_diffusion_offline_1gpu.log).  Every choice gives the same table
# bit for bit.
OFFLINE_CHUNK = 8192
OFFLINE_BLOCK_Q = 128


def check_graph_params(k, gamma):
    """MdirError unless 1 <= k <= 255 and gamma is finite and > 0."""
    if not 1 <= int(k) <= MAX_K:
        raise _lib.MdirError("diffusion needs 1 <= k <= %d neighbours per row (got %d)" % (MAX_K, int(k)))
    if not (math.isfinite(float(gamma)) and float(gamma) > 0):
        raise _lib.MdirError("diffusion needs a finite gamma > 0 (got %r)" % (gamma,))


def check_search_params(k, trunc, k_q, alpha, iters, rtol):
    """MdirError unless 1 <= k <= trunc <= 2048, 1 <= k_q <= trunc, 0 < alpha < 1, 1 <= iters <= 1000 and rtol >= 0."""
    k, trunc, k_q, iters = int(k), int(trunc), int(k_q), int(iters)
    if not 1 <= k <= trunc <= MAX_TRUNC:
        raise _lib.MdirError("diffusion needs 1 <= k <= trunc <= %d (got k=%d, trunc=%d)" % (MAX_TRUNC, k, trunc))
    if not 1 <= k_q <= trunc:
        raise _lib.MdirError("diffusion needs 1 <= k_q <= trunc (got k_q=%d, trunc=%d)" % (k_q, trunc))
    if not 0.0 < float(alpha) < 1.0:
        raise _lib.MdirError("diffusion needs 0 < alpha < 1 (got %r)" % (alpha,))
    if not 1 <= iters <= 1000:
        raise _lib.MdirError("diffusion needs 1 <= iters <= 1000 (got %d)" % iters)
    if not float(rtol) >= 0.0:
        raise _lib.MdirError("diffusion needs rtol >= 0 (got %r)" % (rtol,))


def check_offline_params(width, trunc, alpha, iters, rtol):
    """MdirError unless 1 <= width <= min(trunc, 1024), trunc <= 2048 and the solve's parameters are valid."""
    if not 1 <= int(width) <= MAX_WIDTH:
        raise _lib.MdirError("offline diffusion needs 1 <= width <= %d (got %d)" % (MAX_WIDTH, int(width)))
    check_search_params(width, trunc, 1, alpha, iters, rtol)


def check_combine_params(k, k_q, width):
    """MdirError unless 1 <= k_q <= 128, k_q * width <= 8192 and 1 <= k <= 8192."""
    k, k_q = int(k), int(k_q)
    if not 1 <= k_q <= MAX_KQ:
        raise _lib.MdirError("offline diffusion needs 1 <= k_q <= %d (got %d)" % (MAX_KQ, k_q))
    if k_q * int(width) > MAX_ENTRIES:
        raise _lib.MdirError("offline diffusion needs k_q * width <= %d (got %d * %d)" % (MAX_ENTRIES, k_q, int(width)))
    if not 1 <= k <= MAX_ENTRIES:
        raise _lib.MdirError("offline diffusion needs 1 <= k <= %d (got %d)" % (MAX_ENTRIES, k))


class Diffusion:
    """Diffusion search over a single-GPU Index.

        g = Diffusion(index, k=50, gamma=3.0)      # the graph: one wide search pass per 1,024 rows
        f, ids = g.search(q, k=100, trunc=1000, k_q=10, alpha=0.99, iters=20, rtol=1e-6)
        ids = g.add(vecs); g.remove(ids); g.restore(ids); g.compact()     # the index changes, the graph follows
        tab = g.offline(width=100, trunc=1000)      # DiffusionTable: every row's diffusion, solved once

    The index needs the fp32 master copy and no removed rows among its used slots (call compact() first; a free
    capacity tail is fine).  add / remove / restore / compact through the Diffusion mutate the index and keep the graph
    exactly what a new Diffusion over the live rows would build (DESIGN 2.2e); a mutation made on the Index directly
    makes the graph stale, and search() then raises until a new Diffusion is built.

    State, allocated at the index's capacity (padding past the used slots): the raw lists knn_i / knn_s (the certified
    fp32 top-(k+1) of every slot, -1 / -inf padding for a removed slot), 8 (k + 1) bytes per slot, and the graph nbr /
    S / deg, 8 k + 4 bytes per slot.  update_stats counts, over the life of the object: rows re-searched, pairs passed by
    the bf16 screen, pairs re-scored in fp32, list entries replaced and screen tiles re-run after an overflow."""

    timed = False               # True: update_time gets each update's device time per phase (CUDA events)

    def __init__(self, index, k=50, gamma=3.0):
        check_graph_params(k, gamma)
        if isinstance(index, ShardedIndex) or not isinstance(index, Index):
            raise _lib.MdirError("Diffusion needs a single-GPU Index (a ShardedIndex is not supported)")
        if index.db32 is None:
            raise _lib.MdirError("Diffusion needs the fp32 master copy (keep_fp32=True)")
        n_used = index._n_used
        if not index._live_host[:n_used].all():
            raise _lib.MdirError("Diffusion needs an index without removed rows (%d of %d used slots live): call compact() first"
                                 % (int(index._live_host[:n_used].sum()), n_used))
        self.index, self.k, self.gamma = index, int(k), float(gamma)
        self._version = index._mutations
        self._status = None
        self.update_stats = {"rows_searched": 0, "screen_passed": 0, "rescored": 0, "replaced": 0, "screen_reruns": 0}
        self.update_time = {}
        self._events = []
        cap, dev = index.n, index.device
        with torch.cuda.device(dev):
            self.knn_i = torch.full((cap, self.k + 1), -1, dtype=torch.int32, device=dev)
            self.knn_s = torch.full((cap, self.k + 1), float("-inf"), dtype=torch.float32, device=dev)
            self.nbr = torch.full((cap, self.k), -1, dtype=torch.int32, device=dev)
            self.S = torch.zeros((cap, self.k), dtype=torch.float32, device=dev)
            self.deg = torch.zeros((cap,), dtype=torch.float32, device=dev)
            self._search_rows(torch.arange(n_used, dtype=torch.int64, device=dev))
            self._build_graph()
        self.update_stats["rows_searched"] = 0              # the counters cover the updates

    def graph(self):
        """(nbr (n_used, k) int32 neighbour slots, mutual ones first and -1 padding; S (n_used, k) fp32 normalised
        weights aligned with nbr; deg (n_used,) fp32 degrees), on the device."""
        n = self.index._n_used
        return self.nbr[:n], self.S[:n], self.deg[:n]

    def status(self):
        """Per-query status words of the last search()'s shortlist search (Index.status(): 0 = exact and certified)."""
        return self._status

    def _check_current(self):
        if self.index._mutations != self._version:
            raise _lib.MdirError("the index was mutated (remove / restore / add / compact) after the diffusion graph was built: "
                                 "build a new Diffusion")

    @contextlib.contextmanager
    def _phase(self, name):
        """Brackets one phase of an update with CUDA events when `timed` is set."""
        if not self.timed:
            yield
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        yield
        b.record()
        self._events.append((name, a, b))

    def _finish(self):
        """End of an update: the graph is current again; with `timed`, update_time = ms per phase of this update."""
        self._version = self.index._mutations
        if self.timed:
            torch.cuda.current_stream().synchronize()
            self.update_time = {}
            for name, a, b in self._events:
                self.update_time[name] = self.update_time.get(name, 0.0) + a.elapsed_time(b)
            self._events = []

    def _search_rows(self, slots):
        """The raw lists of these slots (a device int64 tensor), with the build's own call: the certified fp32
        top-(k+1) of each row against the index, DBA_BLOCK rows per search, wide passes."""
        index = self.index
        self.update_stats["rows_searched"] += int(slots.numel())
        with self._phase("search"):
            for r0 in range(0, slots.numel(), DBA_BLOCK):
                b = slots[r0:r0 + DBA_BLOCK]
                s, i = index.search(index.db32[b], self.k + 1, precision="fp32", block_q=WIDE_Q)
                self.knn_s[b] = s
                self.knn_i[b] = i

    def _build_graph(self):
        """nbr / S / deg over the used slots from the raw lists (the build's kernels; padding rows give empty rows)."""
        n_used, lib = self.index._n_used, _lib.lib()
        with self._phase("graph"):
            _lib.check(lib.mdir_diffusion_graph(_lib.ptr(self.knn_i), _lib.ptr(self.knn_s), n_used, self.k, _lib.ptr(self.index.slot_id),
                                                self.gamma, _lib.ptr(self.nbr), _lib.ptr(self.S), _lib.ptr(self.deg), _lib.stream()),
                       "mdir_diffusion_graph")
            _lib.check(lib.mdir_diffusion_normalize(_lib.ptr(self.nbr), _lib.ptr(self.S), _lib.ptr(self.deg), n_used, self.k, _lib.ptr(self.S),
                                                    _lib.stream()), "mdir_diffusion_normalize")

    def _merge_batch(self, bslot, live0, n_target):
        """The reverse merge: the rows of slots bslot (device int64) into the lists of the slots [0, n_target) that are
        set in live0 (the bitmap before the mutation, so the batch itself is no target).  One dense bf16 scan of the
        batch against SCREEN_PLANE_BYTES-sized row chunks, then mdir_diffusion_merge per chunk; the tiles' counts are
        read back once, and a tile that overflowed MERGE_CAP is re-run with exactly the room its count asks for."""
        index, lib = self.index, _lib.lib()
        nb, D = int(bslot.numel()), index.D
        if nb == 0 or n_target == 0:
            return
        dev = index.device
        stats = index.stats()                              # covers every row, the batch included (add merges its stats)
        q16 = index.db16[bslot]
        eps = torch.empty((nb,), dtype=torch.float32, device=dev)
        _lib.check(lib.mdir_diffusion_batch_eps(_lib.ptr(index.db32[bslot]), nb, D, _lib.ptr(stats), _lib.ptr(eps), _lib.stream()),
                   "mdir_diffusion_batch_eps")
        rows = max(MERGE_TILE, SCREEN_PLANE_BYTES // (4 * nb) // MERGE_TILE * MERGE_TILE)
        rows = min(rows, -(-n_target // MERGE_TILE) * MERGE_TILE)
        plane = torch.empty((nb, rows), dtype=torch.float32, device=dev)
        n_tiles = -(-n_target // MERGE_TILE)
        cnt = torch.empty((n_tiles,), dtype=torch.int32, device=dev)
        rep = torch.empty((n_tiles,), dtype=torch.int32, device=dev)

        def run(r0, cap, tiles=None):
            r1 = min(r0 + rows, n_target)
            with self._phase("scan"):
                _lib.check(lib.mdir_sim_scan_dense_bf16(_lib.ptr(index.db16[r0:r1]), r1 - r0, _lib.ptr(q16), nb, D, _lib.ptr(plane), rows,
                                                        _lib.stream()), "mdir_sim_scan_dense_bf16")
            n_run = -(-(r1 - r0) // MERGE_TILE) if tiles is None else int(tiles.numel())
            seg = self._seg(2 * n_run * cap)
            with self._phase("merge"):
                _lib.check(lib.mdir_diffusion_merge(_lib.ptr(plane), rows, nb, r0, r1 - r0, _lib.ptr(tiles), n_run, _lib.ptr(live0),
                                                    _lib.ptr(eps), _lib.ptr(bslot), _lib.ptr(index.db32), D, _lib.ptr(index.slot_id),
                                                    _lib.ptr(self.knn_i), _lib.ptr(self.knn_s), self.k, _lib.ptr(seg), cap, _lib.ptr(cnt),
                                                    _lib.ptr(rep), _lib.stream()), "mdir_diffusion_merge")

        cap = MERGE_CAP
        for r0 in range(0, n_target, rows):
            run(r0, cap)
        c, r = cnt.cpu().numpy(), rep.cpu().numpy()         # the call's synchronisation point
        st = self.update_stats
        st["screen_passed"] += int(c.sum())
        over = np.flatnonzero(c > cap)
        st["rescored"] += int(c.sum() - c[over].sum())
        st["replaced"] += int(r.sum())
        if over.size:
            st["screen_reruns"] += int(over.size)
            cap2 = int(c[over].max())
            for r0 in sorted({int(t) * MERGE_TILE // rows * rows for t in over}):
                t = over[(over * MERGE_TILE >= r0) & (over * MERGE_TILE < r0 + rows)]
                run(r0, cap2, torch.from_numpy(t.astype(np.int32)).to(dev))
            c2, r2 = cnt[torch.from_numpy(over).to(dev)].cpu().numpy(), rep[torch.from_numpy(over).to(dev)].cpu().numpy()
            if (c2 > cap2).any():
                raise _lib.MdirError("diffusion merge re-run overflowed its exact capacity (internal error)")
            st["screen_passed"] += int(c2.sum())
            st["rescored"] += int(c2.sum())
            st["replaced"] += int(r2.sum())

    def _seg(self, n):
        """The reverse merge's candidate segments (uint64), grown on demand and kept."""
        seg = getattr(self, "_seg_buf", None)
        if seg is None or seg.numel() < n:
            seg = self._seg_buf = torch.empty((n,), dtype=torch.int64, device=self.index.device)
        return seg

    def _insert(self, bslot, live0, n_target):
        """Rows that became live (bslot): their own lists, then the reverse merge into everyone else's, then the graph."""
        self._search_rows(bslot)
        self._merge_batch(bslot, live0, n_target)
        self._build_graph()

    def add(self, vecs):
        """index.add(vecs), and the graph follows; returns the new ids.  The new rows' lists come from the build's
        search; every other live row's list takes in the new rows that beat its (k+1)-th entry (the reverse merge: a
        certified bf16 screen of the new rows against the database, exact fp32 re-scores of the pairs that pass).  Cost:
        one search of the new rows plus one dense bf16 scan of them against the used rows, then the graph kernels.
        Errors (a full index, wrong shape) are raised by index.add before anything changes.  Runs on the current stream
        and synchronises with the host: once for the merge's counters, besides the searches' own status checks."""
        self._check_current()
        index = self.index
        s0, live0 = index._n_used, index.live.clone()
        ids = index.add(vecs)
        with torch.cuda.device(index.device):
            if index._n_used > s0:
                self._insert(torch.arange(s0, index._n_used, dtype=torch.int64, device=index.device), live0, s0)
        self._finish()
        return ids

    def restore(self, ids):
        """index.restore(ids), and the graph follows: the restored rows get lists from the build's search and enter the
        other live rows' lists by the reverse merge of add().  Errors (an id never issued, or purged by compact) are
        raised by index.restore before anything changes.  Synchronises with the host as add() does."""
        self._check_current()
        index = self.index
        before, live0 = index._live_host.copy(), index.live.clone()
        index.restore(ids)
        with torch.cuda.device(index.device):
            back = np.flatnonzero(index._live_host & ~before)
            if back.size:
                self._insert(torch.from_numpy(back).to(index.device), live0, index._n_used)
        self._finish()

    def remove(self, ids):
        """index.remove(ids), and the graph follows: the removed rows' lists become padding and their graph rows empty;
        the live rows whose lists held one of them (about k + 1 per removed row) are searched again with the build's
        call.  The cost grows with that number: removing a large fraction of the rows approaches the cost of a rebuild.
        Errors are raised by index.remove before anything changes.  Synchronises with the host once to find the rows to
        search again, besides the searches' own status checks."""
        self._check_current()
        index = self.index
        version = index._mutations
        index.remove(ids)
        if index._mutations != version:
            lib = _lib.lib()
            with torch.cuda.device(index.device):
                n_used = index._n_used
                flag = torch.empty((n_used,), dtype=torch.uint8, device=index.device)
                with self._phase("stale"):
                    _lib.check(lib.mdir_diffusion_stale_rows(_lib.ptr(self.knn_i), _lib.ptr(self.knn_s), n_used, self.k,
                                                             _lib.ptr(index.slot_id), _lib.ptr(index.live), _lib.ptr(flag), _lib.stream()),
                               "mdir_diffusion_stale_rows")
                self._search_rows(torch.nonzero(flag).view(-1))
                self._build_graph()
        self._finish()

    def compact(self):
        """index.compact(), and the graph follows: the live slots' lists move to the front in the same stable order
        (they hold ids, which compaction keeps, so no list changes) and the graph is rebuilt from them.  Returns the
        number of rows purged.  Afterwards graph(), search() and its status words equal those of a new
        Diffusion(index, k, gamma) bit for bit."""
        self._check_current()
        index = self.index
        n_old = index._n_used
        keep = np.flatnonzero(index._live_host[:n_old])
        purged = index.compact()
        if purged:
            with torch.cuda.device(index.device):
                keep_d = torch.from_numpy(keep).to(index.device)
                n = keep.size
                self.knn_i[:n] = self.knn_i[keep_d]
                self.knn_s[:n] = self.knn_s[keep_d]
                self.knn_i[n:n_old] = -1
                self.knn_s[n:n_old] = float("-inf")
                self.nbr[n:n_old] = -1
                self.S[n:n_old] = 0.0
                self.deg[n:n_old] = 0.0
                self._build_graph()
        self._finish()
        return purged

    def search(self, q, k=100, trunc=1000, k_q=10, alpha=0.99, iters=20, rtol=1e-6):
        """q: (N_q, D) fp32 (host or device).  Returns (f (N_q, k) fp32, ids (N_q, k) int32) on the device: the shortlist
        L = index.search(q, trunc, precision="fp32") ranked by (f desc, position in L asc), f the CG solution of
        (I - alpha S_LL) f = y with y_u = max(s_u, 0)^gamma on the first k_q rows of L; -inf / -1 padding past |L|."""
        check_search_params(k, trunc, k_q, alpha, iters, rtol)
        index = self.index
        self._check_current()
        k, trunc = int(k), int(trunc)
        dev = index.device
        with torch.cuda.device(dev):
            q32 = _as_dev_f32(q, dev)
            n_q = q32.shape[0]
            f = torch.empty((n_q, k), dtype=torch.float32, device=dev)
            out = torch.empty((n_q, k), dtype=torch.int32, device=dev)
            if n_q == 0:
                self._status = torch.empty((0,), dtype=torch.int32, device=dev)
                return f, out
            s, ids = index.search(q32, trunc, precision="fp32", check=True)
            self._status = index.status()[:n_q].clone()
            lib = _lib.lib()
            ws_bytes = lib.mdir_diffusion_solve_workspace_bytes(n_q, trunc, self.k)
            ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
            _lib.check(lib.mdir_diffusion_solve(_lib.ptr(ids), _lib.ptr(s), n_q, trunc, _lib.ptr(index.slot_id), index._n_used,
                                                _lib.ptr(self.nbr), _lib.ptr(self.S), self.k, int(k_q), self.gamma, float(alpha),
                                                int(iters), float(rtol), k, _lib.ptr(ws), ws_bytes, _lib.ptr(f), _lib.ptr(out),
                                                _lib.stream()), "mdir_diffusion_solve")
            return f, out

    def offline(self, width=100, trunc=1000, alpha=0.99, iters=20, rtol=1e-6):
        """The offline table (DiffusionTable): every used slot's row diffused as a query with k_q = 1, solved now and
        truncated to its best `width` entries.  The graph must be current.  Cost: one certified fp32 top-trunc search
        of every used row plus one solve per row (DESIGN 2.2e); memory 8 width bytes per slot of the index's capacity."""
        return DiffusionTable(self, width, trunc, alpha, iters, rtol)


class DiffusionTable:
    """Offline diffusion (Yang, Hinami, Matsui, Ly, Satoh, AAAI 2019: diffusion decoupled into online and offline
    processing): diffusion is linear in its right-hand side, so each database row's diffusion is solved once, and a
    query's result is the weighted sum of the table rows of its top-k_q neighbours.  The query needs one top-k_q search
    and one combine kernel, no shortlist of trunc rows and no solve.

        tab = dif.offline(width=100, trunc=1000, alpha=0.99, iters=20, rtol=1e-6)
        f, ids = tab.search(q, k=100, k_q=10)        # device tensors, like Diffusion.search
        tab.status()                                  # status words of the k_q search
        tab_ids, tab_f = tab.table()                  # (n_used, width) views on the device

    Slot i's table row is Diffusion.search(db32[i:i+1], k=width, trunc, k_q=1, alpha, iters, rtol), ids (int32, -1
    padding) and f (fp32, -inf padding) in the solve's order.  The right-hand side is seeded on the row's shortlist's first
    entry: the row itself, or an exact duplicate with a lower id, which then wins the score tie, so both rows get the same
    table row.  Rows are held at the index's capacity; slots past the used ones are padding.

    The table is a snapshot: any mutation of the index after the build, through the Diffusion too (which keeps its graph
    current, not the table), makes search() raise until offline() is run again."""

    timed = False               # True: build_time gets the build's device time of the search passes and the solves (ms)

    def __init__(self, diffusion, width=100, trunc=1000, alpha=0.99, iters=20, rtol=1e-6):
        check_offline_params(width, trunc, alpha, iters, rtol)
        index = diffusion.index
        if isinstance(index, ShardedIndex) or not isinstance(index, Index):
            raise _lib.MdirError("DiffusionTable needs a single-GPU Index (a ShardedIndex is not supported)")
        diffusion._check_current()
        self.index, self.gamma = index, diffusion.gamma
        self.width, self.trunc, self.alpha, self.iters, self.rtol = int(width), int(trunc), float(alpha), int(iters), float(rtol)
        self._version = index._mutations
        self._n_used = index._n_used
        self._status = None
        self.build_time = {}
        dev, lib = index.device, _lib.lib()
        with torch.cuda.device(dev):
            self.tab_ids = torch.full((index.n, self.width), -1, dtype=torch.int32, device=dev)
            self.tab_f = torch.full((index.n, self.width), float("-inf"), dtype=torch.float32, device=dev)
            chunk = int(OFFLINE_CHUNK)
            ws_bytes = lib.mdir_diffusion_solve_workspace_bytes(min(chunk, max(self._n_used, 1)), self.trunc, diffusion.k)
            ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
            events = []
            for r0 in range(0, self._n_used, chunk):
                r1 = min(r0 + chunk, self._n_used)
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if self.timed else None
                if ev:
                    ev[0].record()
                s, L = index.search(index.db32[r0:r1], self.trunc, precision="fp32", block_q=OFFLINE_BLOCK_Q)
                if ev:
                    ev[1].record()
                _lib.check(lib.mdir_diffusion_solve(_lib.ptr(L), _lib.ptr(s), r1 - r0, self.trunc, _lib.ptr(index.slot_id), self._n_used,
                                                    _lib.ptr(diffusion.nbr), _lib.ptr(diffusion.S), diffusion.k, 1, self.gamma, self.alpha,
                                                    self.iters, self.rtol, self.width, _lib.ptr(ws), ws_bytes, _lib.ptr(self.tab_f[r0:r1]),
                                                    _lib.ptr(self.tab_ids[r0:r1]), _lib.stream()), "mdir_diffusion_solve")
                if ev:
                    ev[2].record()
                    events.append(ev)
            if self.timed:
                torch.cuda.current_stream().synchronize()
                self.build_time = {"search": sum(a.elapsed_time(b) for a, b, _ in events),
                                   "solve": sum(b.elapsed_time(c) for _, b, c in events)}

    def table(self):
        """(ids (n_used, width) int32, f (n_used, width) fp32) on the device, row r = slot r at build time."""
        return self.tab_ids[:self._n_used], self.tab_f[:self._n_used]

    def status(self):
        """Per-query status words of the last search()'s k_q search (Index.status(): 0 = exact and certified)."""
        return self._status

    def _check_current(self):
        if self.index._mutations != self._version:
            raise _lib.MdirError("the index was mutated (remove / restore / add / compact) after the diffusion table was built: "
                                 "run offline() again")

    def search(self, q, k=100, k_q=10):
        """q: (N_q, D) fp32 (host or device).  Returns (f (N_q, k) fp32, ids (N_q, k) int32) on the device.  L, s =
        index.search(q, k_q, precision="fp32"); w_u = max(s_u, 0)^gamma; for every id j in the union of the table rows
        of L's slots f_j = sum over u of w_u F[slot(L_u)][j] (fp64, ascending u); the top k by (fp32 f desc, id asc),
        -inf / -1 padding past the union.  Rows outside the union are not candidates."""
        check_combine_params(k, k_q, self.width)
        index = self.index
        self._check_current()
        k, k_q = int(k), int(k_q)
        dev = index.device
        with torch.cuda.device(dev):
            q32 = _as_dev_f32(q, dev)
            n_q = q32.shape[0]
            f = torch.empty((n_q, k), dtype=torch.float32, device=dev)
            out = torch.empty((n_q, k), dtype=torch.int32, device=dev)
            if n_q == 0:
                self._status = torch.empty((0,), dtype=torch.int32, device=dev)
                return f, out
            s, L = index.search(q32, k_q, precision="fp32", check=True)
            self._status = index.status()[:n_q].clone()
            _lib.check(_lib.lib().mdir_diffusion_combine(_lib.ptr(L), _lib.ptr(s), n_q, k_q, _lib.ptr(index.slot_id), index._n_used,
                                                         _lib.ptr(self.tab_ids), _lib.ptr(self.tab_f), self.width, self.gamma, k,
                                                         _lib.ptr(f), _lib.ptr(out), _lib.stream()), "mdir_diffusion_combine")
            return f, out


def _serving_params(source, params):
    """source.search's parameters for captured serving, defaults filled in: (trunc, k_q, alpha, iters, rtol) for a
    Diffusion, (k_q,) for a DiffusionTable."""
    if isinstance(source, Diffusion):
        names = dict(trunc=1000, k_q=10, alpha=0.99, iters=20, rtol=1e-6)
    elif isinstance(source, DiffusionTable):
        names = dict(k_q=10)
    else:
        raise _lib.MdirError("diffusion serving needs a Diffusion or a DiffusionTable (got %s)" % type(source).__name__)
    unknown = sorted(set(params) - set(names))
    if unknown:
        raise TypeError("%s.search() takes no parameter %s" % (type(source).__name__, ", ".join(unknown)))
    return {**names, **params}


class GraphedDiffusion:
    """One diffusion step captured in a CUDA graph: static queries (n_q, D) fp32 in, static f (n_q, k) fp32, ids
    (n_q, k) int32 and status (n_q,) int32 out.

        gd = GraphedDiffusion(dif, n_q=70, k=100, trunc=1000, k_q=10)    # a Diffusion: Diffusion.search's parameters
        gd = GraphedDiffusion(tab, n_q=70, k=100, k_q=10)                # a DiffusionTable: DiffusionTable.search's
        f, ids = gd(q)                                                   # replay on the current stream

    The graph runs the source's own shortlist search, index.search(q, trunc (table: k_q), precision="fp32",
    check=False), copies its status words, then the solve (table: combine) kernel, which reads the used-slot count from
    the index's device copy (Index.n_scan) and the status words from the graph.  A query whose word is nonzero (a
    candidate segment overflowed, or the shortlist was not certified) gets no rows (-inf / -1) and keeps its word: the
    graph has no widening, so whoever owns it redoes those queries with source.search (DiffusionPipeline does).  Every
    other query is bit for bit source.search's row, alone or in any batch (DESIGN 2.2e).

    add / remove / restore / compact made through the Diffusion need no re-capture: the graph reads the index's rows,
    live bitmap, scan extent and slot -> id map and the Diffusion's graph arrays in place.  A replay raises, like
    source.search, once the source is stale: a Diffusion whose index was mutated directly, or a table after any
    mutation (a table's slot -> id lookups use its build-time count)."""

    def __init__(self, source, n_q, k=100, **params):
        p = _serving_params(source, params)
        self.source, self.n_q, self.k, self.params = source, int(n_q), int(k), p
        if not 1 <= self.n_q <= MAX_Q:
            raise _lib.MdirError("GraphedDiffusion: n_q must be in [1, %d] (got %d)" % (MAX_Q, self.n_q))
        online = isinstance(source, Diffusion)
        if online:
            check_search_params(self.k, p["trunc"], p["k_q"], p["alpha"], p["iters"], p["rtol"])
        else:
            check_combine_params(self.k, p["k_q"], source.width)
        source._check_current()
        self.index = index = source.index
        dev, nq, k, lib = index.device, self.n_q, self.k, _lib.lib()
        with torch.cuda.device(dev):
            self.q = torch.zeros((nq, index.D), dtype=torch.float32, device=dev)
            self.f = torch.empty((nq, k), dtype=torch.float32, device=dev)
            self.ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
            self.status = torch.zeros((nq,), dtype=torch.int32, device=dev)
            if online:
                trunc = int(p["trunc"])
                ws_bytes = lib.mdir_diffusion_solve_workspace_bytes(nq, trunc, source.k)
                self._ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)

            def step():
                if online:
                    s, L = index.search(self.q, trunc, precision="fp32", check=False)
                    self.status.copy_(index.status()[:nq])
                    _lib.check(lib.mdir_diffusion_solve_dev(_lib.ptr(L), _lib.ptr(s), nq, trunc, _lib.ptr(index.slot_id), index._n_used,
                                                            _lib.ptr(source.nbr), _lib.ptr(source.S), source.k, int(p["k_q"]), source.gamma,
                                                            float(p["alpha"]), int(p["iters"]), float(p["rtol"]), k, _lib.ptr(self._ws),
                                                            ws_bytes, _lib.ptr(self.f), _lib.ptr(self.ids), _lib.ptr(index.n_scan),
                                                            _lib.ptr(self.status), _lib.stream()), "mdir_diffusion_solve_dev")
                else:
                    s, L = index.search(self.q, int(p["k_q"]), precision="fp32", check=False)
                    self.status.copy_(index.status()[:nq])
                    _lib.check(lib.mdir_diffusion_combine_dev(_lib.ptr(L), _lib.ptr(s), nq, int(p["k_q"]), _lib.ptr(index.slot_id),
                                                              source._n_used, _lib.ptr(source.tab_ids), _lib.ptr(source.tab_f), source.width,
                                                              source.gamma, k, _lib.ptr(self.f), _lib.ptr(self.ids), None,
                                                              _lib.ptr(self.status), _lib.stream()), "mdir_diffusion_combine_dev")
                return s, L

            prof, index.prof = getattr(index, "prof", None), None            # no timing events inside the graph
            try:
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):                             # warm-up: stats, workspaces, kernel attributes
                    step()
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    self._shortlist = step()      # held: the graph writes these buffers on every replay
            finally:
                index.prof = prof

    def _check_current(self):
        self.source._check_current()

    def __call__(self, q=None):
        """Replay on the current stream.  q: (n_q, D) fp32 (host, pinned for an asynchronous copy, or device) copied into
        the static input; None keeps the previous queries.  Returns the static (f, ids); `status` holds the words.
        MdirError, before anything is queued, when the source is stale."""
        self._check_current()
        if q is not None:
            self.q.copy_(q, non_blocking=True)
        self.graph.replay()
        return self.f, self.ids


class DiffusionPipeline(_Pipeline):
    """Host-facing diffusion serving: query batches go up from pinned host buffers, GraphedDiffusion replays back to back
    on one compute stream, and each ticket's (f, ids) and status words come back in pinned buffers, copies and replays
    ordered by events only.

        pipe = DiffusionPipeline(dif, n_q=70, k=100, trunc=1000, k_q=10)      # or (tab, n_q=70, k=100, k_q=10)
        t0 = pipe.submit(q_0)
        t1 = pipe.submit(q_1)
        f, ids = pipe.result(t0)                   # numpy views, valid until `depth` more submits
        pipe.add(vecs); pipe.remove(ids); pipe.restore(ids); pipe.compact()     # a Diffusion source only

    result() is source.search's answer for the whole batch, bit for bit: the queries the graph flagged are redone, alone,
    with source.search on the compute stream and written into the ticket's rows (both kernels are batch-invariant).
    n_recovered counts tickets with such queries, recovered the queries by status bit (a query may count in both).

    Mutations (a Diffusion source) go through the Diffusion's own methods on the compute stream, so its graph stays
    current and no graph is re-captured.  They change the graph arrays and the slot -> id map in place, which a ticket
    redone afterwards would read, so every pending ticket is settled first: waited for and its flagged queries redone
    against the graph it was submitted under.  Tickets submitted before a mutation return the answer before it, later
    ones the answer after it.  compact() refuses while tickets are pending, as in the other pipelines.  A table does
    not follow updates: every mutation method raises."""

    def __init__(self, source, n_q, k=100, depth=2, **params):
        if int(depth) < 1:
            raise _lib.MdirError("DiffusionPipeline: depth must be at least 1 (got %d)" % int(depth))
        self.graphs = [GraphedDiffusion(source, n_q, k, **params) for _ in range(int(depth))]
        self.source, self.params = source, self.graphs[0].params
        # _Pipeline's remove / restore / add / compact call self.index's: the source's, which keep its graph current
        self.index, self.local = source, source.index
        self.n_q, self.k = int(n_q), int(k)
        self.depth, self.overlap = int(depth), False
        dev = self.local.device
        with torch.cuda.device(dev):
            self.compute, self.h2d, self.d2h = (torch.cuda.Stream(device=dev) for _ in range(3))
            self.slots = [{
                "q": torch.empty((self.n_q, self.local.D), dtype=torch.float32).pin_memory(),
                "f": torch.empty((self.n_q, self.k), dtype=torch.float32).pin_memory(),
                "ids": torch.empty((self.n_q, self.k), dtype=torch.int32).pin_memory(),
                "status": torch.empty((self.n_q,), dtype=torch.int32).pin_memory(),
                "up": torch.cuda.Event(), "done": torch.cuda.Event(), "down": torch.cuda.Event(),
                "pending": False, "settled": False} for _ in range(self.depth)]
            torch.cuda.synchronize(dev)
        self.n_submitted = 0
        self.n_recovered = 0            # tickets with at least one query redone eagerly
        self.recovered = {"overflow": 0, "uncertified": 0}     # queries redone, by status bit

    def submit(self, q):
        """q: (n_q, D) fp32 (host or device), copied into the slot's pinned staging buffer here, so the caller may reuse
        it at once.  Returns a ticket for result().  MdirError when the source is stale."""
        t_new = self.n_submitted
        slot, gd = self._free_slot(t_new), self.graphs[t_new % self.depth]
        gd._check_current()
        q = torch.as_tensor(q)
        if tuple(q.shape) != tuple(gd.q.shape):
            raise _lib.MdirError("DiffusionPipeline expects query batches of shape %s" % (tuple(gd.q.shape),))
        slot["q"].copy_(q)
        with torch.cuda.device(self.local.device):
            with torch.cuda.stream(self.h2d):              # this slot's previous replay was collected by result()
                gd.q.copy_(slot["q"], non_blocking=True)
                slot["up"].record()
            caller = torch.cuda.current_stream()
            with torch.cuda.stream(self.compute):
                self.compute.wait_event(slot["up"])
                self.compute.wait_stream(caller)          # updates made on the Diffusion directly, on the caller's stream
                gd.graph.replay()
                slot["done"].record()
            with torch.cuda.stream(self.d2h):
                self.d2h.wait_event(slot["done"])
                for name, src in (("f", gd.f), ("ids", gd.ids), ("status", gd.status)):
                    slot[name].copy_(src, non_blocking=True)
                slot["down"].record()
        slot["pending"], slot["settled"] = True, False
        self.n_submitted += 1
        return t_new

    def _settle(self, slot):
        """Wait for a ticket and redo its flagged queries with source.search on the compute stream, into its rows."""
        slot["down"].synchronize()
        status = slot["status"].numpy()
        flagged = np.flatnonzero(status)
        if flagged.size:
            self.n_recovered += 1
            self.recovered["overflow"] += int(((status & STATUS_OVERFLOW) != 0).sum())
            self.recovered["uncertified"] += int(((status & STATUS_UNCERTIFIED) != 0).sum())
            rows = torch.from_numpy(flagged)
            with torch.cuda.device(self.local.device), torch.cuda.stream(self.compute):
                f, ids = self.source.search(slot["q"][rows], k=self.k, **self.params)
                slot["f"][rows] = f.cpu()
                slot["ids"][rows] = ids.cpu()
        slot["settled"] = True

    def result(self, ticket):
        """Blocks until ticket's result is in host memory -> (f (n_q, k) fp32, ids (n_q, k) int32) numpy views of the
        pinned buffers, valid until `depth` more submits."""
        slot = self._pending_slot(ticket)
        if not slot["settled"]:
            self._settle(slot)
        slot["pending"] = False
        return slot["f"].numpy(), slot["ids"].numpy()

    def _refuse_table(self):
        if isinstance(self.source, DiffusionTable):
            raise _lib.MdirError("DiffusionPipeline over a DiffusionTable: the table does not follow updates; mutate through the "
                                 "Diffusion, run offline() again and build a new pipeline")

    def compact(self):
        """Diffusion.compact() on the compute stream; MdirError while a ticket is pending (see _Pipeline.compact)."""
        self._refuse_table()
        return super().compact()

    def _mutate(self, fn):
        """Settle every pending ticket, then run the source's mutation on the compute stream (after every replay queued
        there).  A DiffusionTable raises."""
        self._refuse_table()
        for sl in self.slots:
            if sl["pending"] and not sl["settled"]:
                self._settle(sl)
        with torch.cuda.device(self.local.device):
            caller = torch.cuda.current_stream()
            self.compute.wait_stream(caller)
            with torch.cuda.stream(self.compute):
                out = fn()
            caller.wait_stream(self.compute)          # the caller's later work sees the updated index and graph
            return out

    def map(self, batches):
        """Generator over an iterable of query batches, keeping `depth` tickets in flight."""
        return self._map(batches, self.submit)
