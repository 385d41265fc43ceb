"""Index.range_search: every live row whose score reaches a per-query threshold, in FAISS's CSR layout.

The fp32 route is judged against fp64 scores computed by torch on the device (a path that shares nothing with the scan,
the gather or the emit): the returned set must equal {live rows with score >= min_score} except for rows whose fp64
score lies within TOL of the threshold, where the fp32 summation order decides (counted and bounded).  The bf16 route is
judged against Index.scores(precision="bf16"), which computes the same bf16-input / fp32-accumulate scores densely, so
that comparison is exact.  Against search() both routes must agree bit for bit.

The R1M-shape test is test_range_r1m_shape (select it alone with -k r1m)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 2e-6           # |fp32 score - fp64 score| on unit rows (two fp32 summation orders differ by ~1e-7 at D <= 2048)


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def _unit(x):
    return x / x.norm(dim=1, keepdim=True)


def build_case(dist, n_db, D, n_q, seed):
    """(db (n_db, D) unit fp32 rows on the device, q (n_q, D)): the generators of test_gpu_certificate.py."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    if dist == "randn":
        db = _unit(torch.randn((n_db, D), device=DEV, generator=g))
    elif dist == "clusters":
        cent = torch.randn((200, D), device=DEV, generator=g)
        c = torch.randint(0, 200, (n_db,), device=DEV, generator=g)
        db = _unit(cent[c] + 0.7 * torch.randn((n_db, D), device=DEV, generator=g))
    elif dist == "near_dup":
        db = _unit(torch.randn((n_db, D), device=DEV, generator=g))
        q = _unit(torch.randn((n_q, D), device=DEV, generator=g))
        pos = torch.randperm(n_db, device=DEV, generator=g)[:n_q * 200].view(n_q, 200)
        for j in range(n_q):                  # 200 near-duplicates per query, all scoring 0.9 +- 3e-3
            nz = torch.randn((200, D), device=DEV, generator=g)
            nz = nz - (nz @ q[j])[:, None] * q[j][None, :]
            db[pos[j]] = _unit(q[j][None, :] + 0.484 * nz / D ** 0.5)
        return db, q
    else:
        raise ValueError(dist)
    src = torch.randperm(n_db, device=DEV, generator=g)[:n_q]
    q = _unit(db[src] + 0.5 * torch.randn((n_q, D), device=DEV, generator=g) / D ** 0.5)
    return db, q


def ref64(db, q):
    """(nq, n_db) fp64 scores on the host."""
    return (q.double() @ db.double().t()).cpu().numpy()


def unpack(lims, sc, ids):
    lims, sc, ids = lims.cpu().numpy(), sc.cpu().numpy(), ids.cpu().numpy()
    assert lims[0] == 0 and (np.diff(lims) >= 0).all() and lims[-1] == sc.size == ids.size
    return [(sc[a:b], ids[a:b].astype(np.int64)) for a, b in zip(lims[:-1], lims[1:])]


def assert_sorted(s, i):
    """(score desc, id asc), no repeated id."""
    assert (np.diff(s) <= 0).all()
    tie = np.diff(s) == 0
    assert (np.diff(i)[tie] > 0).all()
    assert np.unique(i).size == i.size


def check_against(res, ref, m_q, tol, ids_of_slot=None, live=None):
    """res: unpack() list; ref (nq, n_slots) scores by slot; m_q thresholds; ids_of_slot maps slots to ids.
    Returns the number of borderline rows (fp64 score within tol of the threshold) on which the route decided."""
    n_slots = ref.shape[1]
    ids_of_slot = np.arange(n_slots) if ids_of_slot is None else ids_of_slot
    live = np.ones(n_slots, bool) if live is None else live
    border = 0
    for j, (s, i) in enumerate(res):
        assert_sorted(s, i)
        slot = np.searchsorted(ids_of_slot, i)
        assert (ids_of_slot[slot] == i).all() and live[slot].all()
        np.testing.assert_allclose(s, ref[j, slot], rtol=0, atol=tol)
        sure = set(ids_of_slot[live & (ref[j] >= m_q[j] + tol)].tolist())
        maybe = set(ids_of_slot[live & (ref[j] >= m_q[j] - tol)].tolist())
        got = set(i.tolist())
        assert sure <= got <= maybe, (j, len(sure - got), len(got - maybe))
        assert (s >= np.float32(m_q[j])).all()
        border += len(got - sure) + len(maybe - got)
    return border


def kth_scores(ref, ks):
    """Per-query threshold = the ks[j]-th best reference score."""
    return np.array([np.sort(ref[j])[::-1][k - 1] for j, k in enumerate(ks)])


@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
def test_fp32_equals_independent_scores(m, dist):
    db, q = build_case(dist, 60000, 256, 24, {"randn": 1, "clusters": 2, "near_dup": 3}[dist])
    index = m.Index(db, device=DEV)
    ref = ref64(db, q)
    ks = np.geomspace(5, 3000, q.shape[0]).astype(int)
    thr = kth_scores(ref, ks) if dist != "near_dup" else np.full(q.shape[0], 0.9)
    lims, sc, ids = index.range_search(q, torch.from_numpy(thr.astype(np.float32)))
    res = unpack(lims, sc, ids)
    border = check_against(res, ref, thr.astype(np.float32), TOL)
    total = int(lims[-1])
    # each threshold is some row's own score, so every query has at least that row on the border
    assert border <= q.shape[0] + max(2, total // 1000), (border, total)
    assert not index.check_overflow() and index.range_stats["rescans"] == 0
    print("range fp32 %s: %d rows, %d borderline (fp64 within %g of the threshold)" % (dist, total, border, TOL))


def test_bf16_equals_dense_bf16_scores(m):
    db, q = build_case("clusters", 60000, 256, 24, 4)
    index = m.Index(db, device=DEV)
    dense = index.scores(q, precision="bf16").cpu().numpy()
    thr = kth_scores(dense, np.geomspace(3, 2500, q.shape[0]).astype(int)).astype(np.float32)
    lims, sc, ids = index.range_search(q, torch.from_numpy(thr), precision="bf16")
    for j, (s, i) in enumerate(unpack(lims, sc, ids)):
        want = np.flatnonzero(dense[j] >= thr[j])
        order = np.lexsort((want, -dense[j, want]))
        assert np.array_equal(i, want[order]) and np.array_equal(s, dense[j, want[order]])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("D,k", [(256, 100), (2048, 100), (2048, 40)])
def test_equals_search_prefix(m, precision, D, k):
    """The range result equals the prefix of search(q, k) above the threshold, id for id.  Scores are bit-identical
    for bf16, and for fp32 wherever search re-scores the row in a pair (the paired summation order is the one range
    search always uses): at D <= 384, where both of search's orders coincide, and at k = 100 with 70 queries, where the
    2-CTA finalize pairs its whole 128-row shortlist.  At k = 40 (a 64-row shortlist) search re-scores every row alone,
    in another order: from D = 2048 on the last bits may differ, so the thresholds sit in gaps of search's scores
    and the scores must agree to 4 ulps."""
    db, q = build_case("randn", 100000 if D == 256 else 60000, D, 70, 5)
    index = m.Index(db, device=DEV)
    s, i = index.search(q, k, precision=precision)
    s, i = s.cpu().numpy(), i.cpu().numpy()
    exact = precision == "bf16" or D <= 384 or k == 100
    same = total = 0
    for pos in (0, k // 3, k // 2):
        if exact:
            thr = s[:, pos].copy()                          # a row of search's list exactly at the threshold
        else:                                               # the middle of the first gap >= 1e-6 at or after pos
            thr = np.empty(s.shape[0], np.float32)
            for j in range(s.shape[0]):
                g = pos + int(np.flatnonzero(s[j, pos:k - 1] - s[j, pos + 1:k] >= 1e-6)[0])
                thr[j] = (s[j, g] + s[j, g + 1]) / 2
        lims, sc, ids = index.range_search(q, torch.from_numpy(thr), precision=precision)
        for j, (rs, ri) in enumerate(unpack(lims, sc, ids)):
            keep = s[j] >= thr[j]
            assert keep.sum() < k
            assert np.array_equal(ri, i[j][keep]), (precision, D, k, pos, j)
            if exact:
                assert np.array_equal(rs.view(np.uint32), s[j][keep].view(np.uint32)), (precision, D, k, pos, j)
            else:
                assert (np.abs(rs - s[j][keep]) <= 4 * np.spacing(np.abs(s[j][keep]))).all(), (D, k, pos, j)
            same += int((rs.view(np.uint32) == s[j][keep].view(np.uint32)).sum())
            total += rs.size
    print("range vs search %s D=%d k=%d: %d of %d scores bit-identical" % (precision, D, k, same, total))


def test_mutable_index_remove_restore_add_compact(m):
    D, n0, cap = 128, 50000, 60000
    db, q = build_case("randn", n0, D, 16, 6)
    index = m.Index(db, device=DEV, capacity=cap)
    thr = np.float32(0.25)
    base = unpack(*index.range_search(q, float(thr)))
    found = np.unique(np.concatenate([i for _, i in base]))
    assert found.size > 50
    rs = np.random.RandomState(0)
    gone = np.concatenate([found[::3], rs.choice(n0, 5000, replace=False)])
    index.remove(gone)
    after = unpack(*index.range_search(q, float(thr)))
    gone_set = set(gone.tolist())
    for (s0, i0), (s1, i1) in zip(base, after):
        assert not gone_set & set(i1.tolist())
        keep = np.array([x not in gone_set for x in i0.tolist()], bool)
        assert np.array_equal(i1, i0[keep]) and np.array_equal(s1, s0[keep])
    index.restore(gone)
    again = unpack(*index.range_search(q, float(thr)))
    for (s0, i0), (s1, i1) in zip(base, again):
        assert np.array_equal(i0, i1) and np.array_equal(s0, s1)
    # add into capacity: near-copies of the queries are found under their new ids
    new = _unit(q + 0.05 * torch.randn(q.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(7)) / D ** 0.5)
    new_ids = index.add(new).numpy()
    assert new_ids[0] == n0
    added = unpack(*index.range_search(q, float(thr)))
    for j, (s1, i1) in enumerate(added):
        assert new_ids[j] in set(i1.tolist())
        assert i1[0] == new_ids[j]                               # the near-copy is the best match
    # remove some rows, then compact: the same (score, id) list as before compaction
    index.remove(np.concatenate([found[1::4], rs.choice(n0, 20000, replace=False), new_ids[::5]]))
    before = unpack(*index.range_search(q, float(thr)))
    before_bf = unpack(*index.range_search(q, float(thr), precision="bf16"))
    assert index.compact() > 0
    post = unpack(*index.range_search(q, float(thr)))
    post_bf = unpack(*index.range_search(q, float(thr), precision="bf16"))
    for (s0, i0), (s1, i1) in list(zip(before, post)) + list(zip(before_bf, post_bf)):
        assert np.array_equal(i0, i1) and np.array_equal(s0.view(np.uint32), s1.view(np.uint32))
    # against fp64 after compaction: ids through the slot -> id map
    all_rows = torch.cat([db, new])
    ids_of_slot = index._ids
    ref = ref64(all_rows[torch.from_numpy(ids_of_slot).to(DEV)], q)
    check_against(post, ref, np.full(q.shape[0], thr), TOL, ids_of_slot=ids_of_slot)


def test_everything_passes_overflow_rescan_and_large_sort(m):
    """min_score = -inf on 200 k rows: every segment overflows the default capacity, the block is re-scanned at the
    exact one, and each query's 200 k survivors take the group sort + merge."""
    D, n = 128, 200000
    db, q = build_case("randn", n, D, 3, 8)
    index = m.Index(db, device=DEV)
    index.remove(np.arange(0, n, 7))
    live = np.ones(n, bool)
    live[::7] = False
    # check=False: the truncated result is flagged, never silent
    lims, sc, ids = index.range_search(q, float("-inf"), check=False)
    assert index.check_overflow() and (index.status().cpu().numpy() & 1).all()
    assert (np.diff(lims.cpu().numpy()) < live.sum()).all()
    r0 = dict(index.range_stats)
    lims, sc, ids = index.range_search(q, float("-inf"))
    assert not index.check_overflow()
    assert index.range_stats["rescans"] == r0["rescans"] + 1 and index.range_stats["large_sorts"] == r0["large_sorts"] + 3
    res = unpack(lims, sc, ids)
    ref = ref64(db, q)
    for j, (s, i) in enumerate(res):
        assert_sorted(s, i)
        assert np.array_equal(np.sort(i), np.flatnonzero(live))
        np.testing.assert_allclose(s, ref[j, i], rtol=0, atol=TOL)
    # bf16: the same rows with the scan's scores, search(precision="bf16")'s list first
    s_b, i_b = index.search(q, 500, precision="bf16")
    lims, sc, ids = index.range_search(q, float("-inf"), precision="bf16")
    for j, (s, i) in enumerate(unpack(lims, sc, ids)):
        assert_sorted(s, i)
        assert i.size == live.sum()
        assert np.array_equal(i[:500], i_b[j].cpu().numpy()) and np.array_equal(s[:500], s_b[j].cpu().numpy())


def test_massive_ties_overflow(m):
    """60 % of the rows are one identical vector: every candidate segment overflows, > 16,384 rows tie exactly, and
    the ties come out by ascending id."""
    D, n = 128, 100000
    db, q = build_case("randn", n, D, 4, 9)
    g = torch.Generator(device=DEV).manual_seed(10)
    dup_rows = torch.randperm(n, device=DEV, generator=g)[:60000]
    db[dup_rows] = q[0]
    index = m.Index(db, device=DEV)
    ref = ref64(db, q)
    thr = np.array([0.5, 0.2, 0.5, 2.0], np.float32)
    r0 = index.range_stats["rescans"]
    res = unpack(*index.range_search(q, torch.from_numpy(thr)))
    assert index.range_stats["rescans"] == r0 + 1 and not index.check_overflow()
    s0, i0 = res[0]
    dups = np.sort(dup_rows.cpu().numpy())
    assert i0.size >= 60000 and np.array_equal(i0[:60000], dups)       # one score, ids ascending
    assert (s0[:60000] == s0[0]).all()
    check_against(res, ref, thr, TOL)
    assert res[3][1].size == 0


def test_ragged_per_query_results(m):
    """Per-query thresholds in one call: none, a few, many (> 16,384), everything, above every score; more than 128
    queries, so two blocks are concatenated into one CSR result."""
    D, n, nq = 128, 100000, 300
    db, q = build_case("clusters", n, D, nq, 11)
    index = m.Index(db, device=DEV)
    ref = ref64(db, q)
    thr = kth_scores(ref, np.full(nq, 40)).astype(np.float32)
    thr[0] = 1.5                                   # above every score
    thr[1] = np.float32(np.sort(ref[1])[::-1][2])  # three rows
    thr[2] = np.float32(np.sort(ref[2])[::-1][30000])   # > 16,384
    thr[3] = -np.inf                               # everything
    thr[200] = np.float32(np.sort(ref[200])[::-1][20000])   # > 16,384, second block
    thr[299] = 2.0
    lims, sc, ids = index.range_search(q, torch.from_numpy(thr))
    res = unpack(lims, sc, ids)
    counts = np.diff(lims.cpu().numpy())
    assert counts[0] == 0 and counts[299] == 0 and counts[3] == n
    assert 2 <= counts[1] <= 4 and counts[2] > 16384 and counts[200] > 16384
    border = check_against(res, ref, thr, TOL)
    assert border <= nq + 10                       # every threshold is a row's own score: that row is on the border
    # the same queries one at a time give the same segments
    for j in (1, 2, 3, 150, 200, 299):
        one = unpack(*index.range_search(q[j:j + 1], float(thr[j])))[0]
        assert np.array_equal(one[1], res[j][1]) and np.array_equal(one[0], res[j][0])


def test_edge_cases(m):
    db, q = build_case("randn", 20000, 64, 5, 12)
    index = m.Index(db, device=DEV)
    lims, sc, ids = index.range_search(q[:0], 0.5)
    assert lims.shape == (1,) and int(lims[0]) == 0 and sc.numel() == 0 and ids.numel() == 0
    lims, sc, ids = index.range_search(q, 1.01)                # above every score of unit rows
    assert (lims.cpu() == 0).all() and sc.numel() == 0
    with pytest.raises(m.MdirError):
        index.range_search(q, float("nan"))
    with pytest.raises(m.MdirError):
        index.range_search(q, torch.tensor([0.1, 0.2, float("nan"), 0.3, 0.4]))
    with pytest.raises(m.MdirError):
        index.range_search(q, torch.zeros(4))
    with pytest.raises(m.MdirError):
        m.Index(db, device=DEV, keep_fp32=False).range_search(q, 0.1)
    # bf16 works without the fp32 master copy
    lims, _, _ = m.Index(db, device=DEV, keep_fp32=False).range_search(q, 0.1, precision="bf16")
    assert lims.shape == (6,)
    # every row removed, and an index with only free capacity
    index.remove(np.arange(20000))
    lims, sc, ids = index.range_search(q, float("-inf"))
    assert lims.shape == (6,) and (lims.cpu() == 0).all() and sc.numel() == 0
    empty = m.Index(db[:1], device=DEV, capacity=1000)
    empty.remove([0])
    assert (empty.range_search(q, float("-inf"))[0].cpu() == 0).all()
    # a range call leaves search() unchanged: its candidate buffers are the range route's own
    index.restore(np.arange(20000))
    s1, i1 = index.search(q, 10)
    index.range_search(q, float("-inf"))
    s2, i2 = index.search(q, 10)
    assert torch.equal(s1, s2) and torch.equal(i1, i2)


def test_range_r1m_shape(m):
    """1,001,001 x 2048, 70 queries, thresholds giving ~100 - 5,000 matches per query: the complete result against the
    fp64 scores of every row."""
    n_db, D, nq = 1001001, 2048, 70
    g = torch.Generator(device=DEV).manual_seed(13)
    db = torch.empty((n_db, D), dtype=torch.float32, device=DEV)
    for r0 in range(0, n_db, 65536):
        r1 = min(n_db, r0 + 65536)
        db[r0:r1] = _unit(torch.randn((r1 - r0, D), device=DEV, generator=g))
    src = torch.randperm(n_db, device=DEV, generator=g)[:nq]
    q = _unit(db[src] + 0.5 * torch.randn((nq, D), device=DEV, generator=g) / D ** 0.5)
    index = m.Index.from_packed(m.search.pack_bf16(db), db32=db)
    ks = np.geomspace(100, 5000, nq).astype(int)
    ref = np.empty((nq, n_db))
    for r0 in range(0, n_db, 200000):
        r1 = min(n_db, r0 + 200000)
        ref[:, r0:r1] = (q.double() @ db[r0:r1].double().t()).cpu().numpy()
    thr = kth_scores(ref, ks).astype(np.float32)
    lims, sc, ids = index.range_search(q, torch.from_numpy(thr))
    res = unpack(lims, sc, ids)
    border = check_against(res, ref, thr, TOL)
    counts = np.diff(lims.cpu().numpy())
    assert ((counts >= ks - 5) & (counts <= ks + 5)).all()
    assert border <= 2 * nq and not index.check_overflow()     # the row at each threshold + ~0.6 more per query at D = 2048
    print("R1M range: %d rows over %d queries, %d borderline, stats %s" % (int(lims[-1]), nq, border, index.range_stats))


def test_writes_stay_inside_their_slices(m):
    """Every kernel of the route writes only where it owns: the gather inside its chunk's survivor slice (the rest of
    the slice keeps a sentinel), the emit / merge each output position exactly once (no position keeps its sentinel,
    none is written twice: ids unique).  Two ordinary queries and two with > 16,384 survivors (group sort + merge);
    check=False keeps the pass on the route's cached buffers, whose tails are inspected."""
    D, n = 128, 60000
    db, q = build_case("randn", n, D, 4, 14)
    index = m.Index(db, device=DEV)
    thr = torch.tensor([0.2, float("-inf"), 0.15, float("-inf")])
    index.range_search(q, thr, check=False)                    # allocates the cached buffers
    surv = index._buf("range_surv", (128, m.search.range_chunks(m.search.RANGE_CAP_L) * m.search.RANGE_CHUNK), torch.int64)
    sentinel = 0x5A5A5A5A5A5A5A5A
    surv.fill_(sentinel)
    lims, sc, ids = index.range_search(q, thr, check=False)
    n_chunks = m.search.range_chunks(m.search.RANGE_CAP_L)
    runs = index._buf("range_runs", (128 * (n_chunks + 1),), torch.int32)[:4 * n_chunks].view(4, n_chunks).cpu().numpy()
    sv = surv[:4].cpu().numpy().reshape(4, n_chunks, m.search.RANGE_CHUNK)
    counts = np.diff(lims.cpu().numpy())
    assert counts[1] > 16384 and counts[3] > 16384 and counts[0] <= 16384 and counts[2] <= 16384
    for j in (0, 2):                                          # the emit only reads these slices: the gather's writes
        for c in range(n_chunks):
            assert (sv[j, c, runs[j, c]:] == sentinel).all(), (j, c)
            assert (sv[j, c, :runs[j, c]] != sentinel).all(), (j, c)
    for j in (1, 3):                                          # group sort in place: each group's keys contiguous
        for g0 in range(0, n_chunks, 16):
            glen = int(runs[j, g0:g0 + 16].sum())
            flat = sv[j, g0:g0 + 16].reshape(-1)
            assert (np.diff(np.ascontiguousarray(flat[:glen]).view(np.uint64)) > 0).all()
    # the outputs: written exactly once each (a kept sentinel would break the unique ids / the order)
    res = unpack(lims, sc, ids)
    for s, i in res:
        assert_sorted(s, i)
        assert (i >= 0).all() and (i < n).all()
