"""The int8 first pass of the certified fp32 search (Index._i8_route): mdir_pack_stats_i8 -> mdir_pack_q_i8 ->
mdir_sim_scan_fused_i8 -> mdir_topk_finalize_rescore_eps.

The first pass scores int8 database rows (per-row scale) against the query as two int8 planes (hi + lo residual);
the finalize re-scores in fp32 every candidate within the per-query bound eps of the k-th fp32 score.  What makes the
answer identical to the bf16 route's is that bound: checked here against every (row, query) pair, then end to end at
the headline size, plus the route choice and the recovery of a flagged block through the bf16 route."""
import numpy as np
import pytest
import torch

from oracle import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def _quant(v, s):
    """numpy restatement of quant_i8 (csrc/topk.cu): rint(v / s) in fp32, half to even, clamped to [-127, 127]."""
    if s <= 0:
        return np.zeros_like(v)
    return np.clip(np.rint(v / np.float32(s)), -127, 127).astype(np.float32)


def _pack_q_numpy(q):
    """-> (hi, lo) int8 planes and (s_hi, s_lo) per query, the arithmetic of pack_q_i8_kernel."""
    hi, lo, sc = [], [], []
    for v in q.astype(np.float32):
        s_hi = np.float32(np.abs(v).max()) / np.float32(127)
        h = _quant(v, s_hi)
        r = (v.astype(np.float64) - np.float64(s_hi) * h).astype(np.float32)      # fmaf(-s_hi, h, v): one rounding
        s_lo = np.float32(np.abs(r).max()) / np.float32(127)
        hi.append(h)
        lo.append(_quant(r, s_lo))
        sc.append((s_hi, s_lo))
    return np.array(hi, np.int8), np.array(lo, np.int8), np.array(sc, np.float32)


def _pack_q(m, index, q):
    lib, _lib = m.lib(), m._lib
    nq, D = q.shape
    n_pad = -(-nq // 16) * 16
    q8 = torch.full((2 * n_pad, D), 99, dtype=torch.int8, device=DEV)
    qsc = torch.empty((nq, 2), dtype=torch.float32, device=DEV)
    qeps = torch.empty((nq,), dtype=torch.float32, device=DEV)
    qd = torch.from_numpy(np.ascontiguousarray(q, dtype=np.float32)).to(DEV)
    _lib.check(lib.mdir_pack_q_i8(_lib.ptr(qd), nq, D, _lib.ptr(index.stats()), _lib.ptr(q8), _lib.ptr(qsc), _lib.ptr(qeps), _lib.stream()))
    torch.cuda.synchronize()
    return q8, qsc, qeps.cpu().numpy().astype(np.float64), n_pad


def _key_scores(keys):
    """key_score (csrc/common.cuh) of uint64 keys -> (fp32 scores, row indices)."""
    o = ~(keys >> np.uint64(32)).astype(np.uint32)
    u = np.where(o >> np.uint32(31) != 0, o ^ np.uint32(0x80000000), o ^ np.uint32(0xffffffff)).astype(np.uint32)
    return u.view(np.float32), (keys & np.uint64(0xffffffff)).astype(np.int64)


@pytest.fixture
def small_shards(m, monkeypatch):
    """Lift the int8 route's minimum shard size for tests whose databases are small."""
    monkeypatch.setattr(m.search, "I8_MIN_ROWS", 0)


def test_query_pack_matches_numpy(m):
    """The two query planes and their scales bit for bit, padding rows zero."""
    db = synth.descriptors(2000, 256, 3)
    q = synth.descriptors(37, 256, 4)
    q[5] *= 0.01                                                        # scales are per query
    index = m.Index(db, device=DEV)
    q8, qsc, _, n_pad = _pack_q(m, index, q)
    q8, qsc = q8.cpu().numpy(), qsc.cpu().numpy()
    hi, lo, sc = _pack_q_numpy(q)
    assert np.array_equal(q8[:37], hi) and np.array_equal(q8[n_pad:n_pad + 37], lo)
    assert not q8[37:n_pad].any() and not q8[n_pad + 37:].any()
    assert np.array_equal(qsc, sc)


@pytest.mark.parametrize("clusters", [0, 40])
def test_int8_bound_holds_and_is_not_vacuous(m, small_shards, clusters):
    """|int8-path score - exact score| <= eps for EVERY (row, query) pair, and eps is within ~100x of the observed error.
    The int8-path scores are the exact restatement of the scan's arithmetic; the scores the fused int8 scan itself
    produced (read back from its candidate keys) match that restatement within the conversion term, and every row the
    restatement puts above the scan's threshold is among its candidates."""
    db = synth.descriptors(60000, 512, 5, clusters=clusters)
    q, _ = synth.planted_queries(db, 64, 6)
    index = m.Index(db, device=DEV)
    st = index.stats().cpu().numpy().astype(np.float64)
    assert index.db8 is not None
    x8 = index.db8.cpu().numpy()
    s_r = index.row_scale.cpu().numpy()
    # the database plane: numpy restatement of pack_stats_i8_kernel, and the residual terms of stats
    want = np.stack([_quant(row, s) for row, s in zip(db, np.abs(db).max(1).astype(np.float32) / np.float32(127))])
    assert np.array_equal(x8, want.astype(np.int8))
    resid = db.astype(np.float64) - s_r[:, None].astype(np.float64) * x8
    e2 = (resid ** 2).sum(1)
    assert e2.max() <= st[2] <= 1.01 * e2.max()
    assert (e2 / (db.astype(np.float64) ** 2).sum(1)).max() <= st[3]
    q8_d, qsc_d, eps, n_pad = _pack_q(m, index, q)
    q8, qsc = q8_d.cpu().numpy(), qsc_d.cpu().numpy()
    nq = q.shape[0]
    # the scan's arithmetic, exact: s_r * (s_hi * <x8, hi> + s_lo * <x8, lo>) (its fp32 rounding is inside eps)
    acc_hi = x8.astype(np.int64) @ q8[:nq].astype(np.int64).T
    acc_lo = x8.astype(np.int64) @ q8[n_pad:n_pad + nq].astype(np.int64).T
    s8 = s_r[:, None].astype(np.float64) * (qsc[:, 0].astype(np.float64) * acc_hi + qsc[:, 1].astype(np.float64) * acc_lo)
    exact = db.astype(np.float64) @ q.astype(np.float64).T
    err = np.abs(s8 - exact).max(axis=0)
    assert np.all(err <= eps), (err.max(), eps.min())
    assert np.all(eps <= 100 * err) and eps.max() < 0.03, (err.max(), eps.max())
    # ---- the fused int8 scan: its candidate keys carry the scores it computed
    S = m.search
    lib, _lib = m.lib(), m._lib
    tau, cand, cnt = index._cand_bufs(nq)
    _lib.check(lib.mdir_sim_scan_fused_i8(_lib.ptr(index.db8), _lib.ptr(index.row_scale), index.n, _lib.ptr(q8_d), _lib.ptr(qsc_d), nq, index.D,
                                          128, _lib.ptr(tau), 0, _lib.ptr(cand), _lib.ptr(cnt), 0, S.FUSED_CAP_L, _lib.ptr(index._fused_ws()),
                                          _lib.stream()), "mdir_sim_scan_fused_i8")
    torch.cuda.synchronize()
    row_len = 148 * S.FUSED_CAP_L                      # the candidate row pitch of the one-launch route (no select segment)
    flat = cand.view(-1)[:nq * row_len].cpu().numpy().view(np.uint64).reshape(nq, row_len)
    counts = cnt[:nq].cpu().numpy().astype(np.int64)
    assert counts[:, 0].max() == 0 and counts.max() <= S.FUSED_CAP_L
    tau_s, _ = _key_scores(tau[:nq].cpu().numpy().view(np.uint64))
    # per (row, query): s_r * (s_hi * acc_hi + s_lo * acc_lo) evaluated in fp32 -- a few roundings of its two terms
    conv = 8 * 2.0 ** -24 * np.abs(s_r)[:, None] * (np.abs(qsc[:, 0] * acc_hi) + np.abs(qsc[:, 1] * acc_lo))
    for j in range(nq):
        keys = np.concatenate([flat[j, c * S.FUSED_CAP_L:c * S.FUSED_CAP_L + counts[j, 1 + c]] for c in range(148)])
        got, rows = _key_scores(keys)
        assert len(rows) > 128 and len(np.unique(rows)) == len(rows)
        assert np.all(np.abs(got - s8[rows, j]) <= conv[rows, j] + 1e-12), np.abs(got - s8[rows, j]).max()
        must = np.nonzero(s8[:, j] > float(tau_s[j]) + conv[:, j])[0]       # above the threshold whatever the rounding
        assert np.isin(must, rows).all(), (j, len(must), len(rows))


def _unit(x):
    return x / x.norm(dim=1, keepdim=True)


def _r1m(dist, seed, n_db=1001001, D=2048, n_q=70):
    g = torch.Generator(device=DEV).manual_seed(seed)
    db = torch.empty((n_db, D), dtype=torch.float32, device=DEV)
    cent = torch.randn((1000, D), device=DEV, generator=g) if dist == "clusters" else None
    for r0 in range(0, n_db, 65536):
        n = min(65536, n_db - r0)
        x = torch.randn((n, D), device=DEV, generator=g)
        if cent is not None:
            x = cent[torch.randint(0, 1000, (n,), device=DEV, generator=g)] + 0.7 * x
        db[r0:r0 + n] = _unit(x)
    q = _unit(torch.randn((n_q, D), device=DEV, generator=g))
    if dist == "near_dup":                      # 200 rows per query at 0.9 +- 3e-3
        pos = torch.randperm(n_db, device=DEV, generator=g)[:n_q * 200].view(n_q, 200)
        for j in range(n_q):
            nz = torch.randn((200, D), device=DEV, generator=g)
            nz = nz - (nz @ q[j])[:, None] * q[j][None, :]
            db[pos[j]] = _unit(q[j][None, :] + 0.484 * nz / D ** 0.5)
    else:
        src = torch.randperm(n_db, device=DEV, generator=g)[:n_q]
        q = _unit(db[src] + 0.5 * torch.randn((n_q, D), device=DEV, generator=g) / D ** 0.5)
    return db, q


@pytest.mark.parametrize("dist", ["randn", "clusters", "near_dup"])
def test_r1m_int8_route_equals_bf16_route(m, dist):
    """The headline shape: the int8 route's certified top-100 is bit-identical to the bf16 route's."""
    db, q = _r1m(dist, {"randn": 51, "clusters": 52, "near_dup": 53}[dist])
    index = m.Index.from_packed(m.search.pack_bf16(db), db32=db)
    s8, i8 = index.search(q, 100, precision="fp32")
    assert index.route == "int8" and index.cert["int8_blocks"] == 1, index.cert
    db8, rs = index.db8, index.row_scale
    index.db8 = None                                                   # no int8 plane: the bf16 route
    s16, i16 = index.search(q, 100, precision="fp32")
    assert index.route == "bf16"
    index.db8, index.row_scale = db8, rs
    assert torch.equal(i8, i16) and torch.equal(s8, s16)
    assert index.cert["uncertified"] == 0 and not bool(index.status().any().item())
    print("R1M %s: int8 route counters %s" % (dist, index.cert))


def test_small_shard_stays_on_bf16(m):
    """Below I8_MIN_ROWS the int8 bound would not clear the fused scan's threshold: no int8 plane, bf16 route."""
    db = synth.descriptors(100000, 256, 21)
    index = m.Index(db, device=DEV)
    index.search(synth.descriptors(8, 256, 22), 100, precision="fp32")
    assert index.n < m.search.I8_MIN_ROWS and index.db8 is None and index.route == "bf16"


def test_heavy_tailed_database_stays_on_bf16(m, small_shards):
    """A few dimensions x20: the int8 residual is too large against the rows, so the shard keeps the bf16 first pass
    (and no int8 plane), and the answer is still the exact ranking."""
    db = synth.descriptors(100000, 256, 11)
    db[:, :4] *= 20
    db /= np.linalg.norm(db, axis=1, keepdims=True)
    q = synth.descriptors(16, 256, 12)
    index = m.Index(db, device=DEV)
    s, i = index.search(q, 100, precision="fp32")
    assert index.route == "bf16" and index.db8 is None and index.cert["int8_blocks"] == 0
    assert index._fused_ok(128, 16)                                   # the bf16 route is the fused one: only the residual decided
    exact = q.astype(np.float64) @ db.astype(np.float64).T
    order = np.lexsort((np.broadcast_to(np.arange(db.shape[0]), exact.shape), -exact), axis=1)[:, :100]
    got = i.cpu().numpy()
    for j in range(16):                                                # swaps only inside fp32 noise
        diff = got[j] != order[j]
        assert np.all(np.abs(exact[j, got[j][diff]] - exact[j, order[j][diff]]) <= 2e-6)


def test_flagged_int8_block_recovers_through_bf16(m, small_shards):
    """600 near-ties per query at D = 2048: more rows within the int8 bound than the extension area of this shard
    holds, so the int8 block is flagged; search(check=True) redoes it through the bf16 route, which widens until
    certified, and the answer is the exact ranking."""
    n_db, D, n_q, k, dup = 120000, 2048, 6, 100, 600
    rs = np.random.RandomState(13)
    db = synth.descriptors(n_db, D, 14)
    q = synth.descriptors(n_q, D, 15)
    pos = rs.permutation(n_db)[:n_q * dup].reshape(n_q, dup)
    for j in range(n_q):
        nz = rs.randn(dup, D).astype(np.float32)
        nz -= (nz @ q[j])[:, None] * q[j][None, :]
        v = q[j][None, :] + 0.1 * nz / np.sqrt(D)
        db[pos[j]] = v / np.linalg.norm(v, axis=1, keepdims=True)
    index = m.Index(db, device=DEV)
    index.search(q, k, precision="fp32", check=False)
    assert index.route == "int8" and index.check_overflow()
    s, i = index.search(q, k, precision="fp32")
    assert index.cert["int8_redone"] == 1 and index.route == "bf16" and index.cert["uncertified"] == 0, index.cert
    exact = q.astype(np.float64) @ db.astype(np.float64).T
    order = np.lexsort((np.broadcast_to(np.arange(n_db), exact.shape), -exact), axis=1)[:, :k]
    got = i.cpu().numpy()
    for j in range(n_q):
        diff = got[j] != order[j]
        assert np.all(np.abs(exact[j, got[j][diff]] - exact[j, order[j][diff]]) <= 2e-6)
        assert np.all(np.abs(s.cpu().numpy()[j] - exact[j, order[j]]) <= 2e-6)
