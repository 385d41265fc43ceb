"""Host side of Index.compact (no GPU): the chunk schedule of the in-place move, and the slot -> id bookkeeping of
remove / restore / add / compact on the index's host mirrors."""
import numpy as np
import pytest

from mdir_b200 import _lib
from mdir_b200.search import Index, compaction_schedule


def _replay(live, chunk):
    """Run the schedule on a model of the planes: a chunk reads all its live rows (staged: every read before any write;
    direct: reads and writes interleaved, so they must be disjoint), then writes their destinations.  Asserts that no
    row is read after it was overwritten and returns the final row -> slot contents."""
    live = np.asarray(live, dtype=bool)
    slots = np.arange(live.size)                  # slot s holds row s
    written = np.zeros(live.size, dtype=bool)
    prev_hi = 0
    for lo, hi, dst0, n_dst, staged in compaction_schedule(live, chunk):
        assert lo >= prev_hi and hi - lo <= chunk        # ascending, disjoint chunks
        prev_hi = hi
        src = lo + np.flatnonzero(live[lo:hi])
        assert len(src) == n_dst and dst0 == int(live[:lo].sum())
        dst = np.arange(dst0, dst0 + n_dst)
        assert not written[src].any()                   # nothing read after being overwritten
        assert (dst <= src).all() and dst0 + n_dst <= hi
        if not staged:
            assert dst0 + n_dst <= lo and not np.intersect1d(src, dst).size
        vals = slots[src].copy()
        slots[dst] = vals
        written[dst] = True
    return slots


CASES = {
    "nothing_removed": lambda n, rs: np.ones(n, dtype=bool),
    "all_removed": lambda n, rs: np.zeros(n, dtype=bool),
    "head": lambda n, rs: np.arange(n) >= n // 3,
    "tail": lambda n, rs: np.arange(n) < n - n // 3,
    "one_dead_first": lambda n, rs: np.arange(n) != 0,
    "one_dead_last": lambda n, rs: np.arange(n) != n - 1,
    "random_10": lambda n, rs: rs.rand(n) > 0.10,
    "random_50": lambda n, rs: rs.rand(n) > 0.50,
    "random_99": lambda n, rs: rs.rand(n) > 0.99,
    "runs": lambda n, rs: (np.arange(n) // 37) % 3 != 1,
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("n", [1, 31, 33, 255, 257, 1000, 3001])
@pytest.mark.parametrize("chunk", [1, 7, 32, 100, 256, 4096])
def test_schedule_never_reads_an_overwritten_row(case, n, chunk):
    rs = np.random.RandomState(n * 31 + chunk)
    live = CASES[case](n, rs)
    slots = _replay(live, chunk)
    keep = np.flatnonzero(live)
    assert np.array_equal(slots[:keep.size], keep)      # stable: live rows in their order at the front
    if live.all():
        assert compaction_schedule(live, chunk) == []


def test_schedule_uses_direct_moves_once_enough_rows_are_dead():
    live = np.arange(100000) % 2 == 0
    sched = compaction_schedule(live, 1000)
    assert sched[0][4] and not any(c[4] for c in sched[2:])


def _host_index(n, cap, base):
    """An Index with only its host mirrors (the bookkeeping under test); device updates are replaced by the mirror update
    they accompany."""
    ix = Index.__new__(Index)
    ix.idx_base, ix.n = base, cap
    ix._live_host = np.zeros(cap, dtype=bool)
    ix._live_host[:n] = True
    ix._n_used = n
    ix._ids = np.arange(base, base + n, dtype=np.int64)
    ix._next_id = n
    ix.device = None
    return ix


class _NoDevice:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


@pytest.fixture
def host_only(monkeypatch):
    import torch

    def set_live(self, rows, value):
        self._live_host[np.unique(rows)] = bool(value)

    def add(self, m):                                    # Index.add without its device writes
        s0 = self._n_used
        assert s0 + m <= self.n
        ids = self._issue_ids(m)
        self._live_host[s0:s0 + m] = True
        return ids

    def compact(self):                                   # Index.compact without its device launches
        self._compacted_mirrors(np.flatnonzero(self._live_host[:self._n_used]))

    monkeypatch.setattr(Index, "_set_live", set_live)
    monkeypatch.setattr(torch.cuda, "device", lambda d: _NoDevice())
    return add, compact


def test_ids_survive_repeated_compactions(host_only):
    add, compact = host_only
    base = 500
    ix = _host_index(1000, 1200, base)
    model = {base + s: True for s in range(1000)}       # id -> live
    rs = np.random.RandomState(1)
    for rnd in range(4):
        live_ids = np.array(sorted(i for i, v in model.items() if v))
        gone = rs.choice(live_ids, live_ids.size // 3, replace=False)
        ix.remove(gone)
        for g in gone:
            model[int(g)] = False
        ix.remove(gone[:5])                               # removing a removed id: no-op
        compact(ix)
        purged = [int(g) for g in gone]
        for g in purged:
            del model[g]
        with pytest.raises(_lib.MdirError, match="purged"):
            ix.restore(purged[:1])
        ix.remove(purged[:4])                             # removing a purged id: no-op
        assert np.array_equal(ix._ids, np.array(sorted(model)))
        assert (np.diff(ix._ids) > 0).all()               # strictly increasing: searchsorted finds every slot
        _, pos, found = ix._slots(np.array(sorted(model)))
        assert found.all() and np.array_equal(pos, np.arange(len(model)))
        new = add(ix, 200)
        assert new[0] == base + 1000 + 200 * rnd         # ids continue from the highest issued, never reused
        for i in new:
            model[int(i)] = True
        # remove + restore of a live id round-trips
        some = new[:3]
        ix.remove(some)
        assert not ix._live_host[ix._slots(some)[1]].any()
        ix.restore(some)
        assert ix._live_host[ix._slots(some)[1]].all()
    assert ix._next_id == 1800 and int(ix._ids.max()) >= base + ix.n        # ids now exceed idx_base + capacity
    with pytest.raises(_lib.MdirError, match="outside"):
        ix.restore([base + 1800])                         # past every id issued
    with pytest.raises(_lib.MdirError, match="outside"):
        ix.remove([base - 1])
    with pytest.raises(_lib.MdirError, match="outside"):
        ix.remove([base + 1800 + 10 ** 6])


def test_restore_before_any_compaction_keeps_its_errors(host_only):
    ix = _host_index(3000, 3100, 1000)
    with pytest.raises(_lib.MdirError, match="never filled"):
        ix.restore([4000])                                # a free slot was never filled
    ix.remove([1000, 1000, 1001])
    assert ix._live_host.sum() == 2998
    ix.restore([1000])
    assert ix._live_host.sum() == 2999
    with pytest.raises(_lib.MdirError):
        ix.remove([999])
