"""Three-tier certified re-score of the int8 route (mdir_topk_finalize_rescore_tiered_ids, Index.tiered).

The extension E of the int8 certificate (candidates with s8 >= t0 - eps8 outside the shortlist S) is re-scored from
the bf16 rows first; only the rows F of E with s16 >= t0 - eps16 are re-scored in fp32.  The answer must be the two-tier
one (Index.tiered = False) bit for bit, status words included, and the exact fp32 top-k: both finalizes run here on
the same int8 first-pass output and are judged against an independent dense 3xTF32 -> fp64 ranking.  Also: F is
actually used (rows outside S reach the answer), the tier-2 bound holds on measured scores, and search's fp32 scores
equal range_search's bit for bit (one summation order for every re-scored row)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N_R1M, D_R1M, NQ, K = 1001001, 2048, 70, 100


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def _unit(x):
    return x / x.norm(dim=1, keepdim=True)


def _fill(db, gen, make_block, step=65536):
    for r0 in range(0, db.shape[0], step):
        n = min(step, db.shape[0] - r0)
        db[r0:r0 + n] = make_block(n, gen)


def build_case(dist, n_db, D, n_q, seed, dup_per_query=200):
    """(db (n_db, D) unit fp32 rows on the device, q (n_q, D)).  randn queries are bench.py's kind (unit randn,
    unrelated to the rows); clusters: 1k Gaussian clusters; near_dup: dup_per_query rows per query at 0.9 +- 3e-3;
    straddle: per query 400 rows spread evenly over 0.9 +- 5e-5 (far inside the int8 score noise, so the int8 shortlist
    holds a random third of them and t0 falls among them) and 100 rows at 0.895 (inside eps8, outside eps16)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    db = torch.empty((n_db, D), dtype=torch.float32, device=DEV)
    if dist == "clusters":
        cent = torch.randn((1000, D), device=DEV, generator=g)

        def blk(n, gen):
            c = torch.randint(0, 1000, (n,), device=DEV, generator=gen)
            return _unit(cent[c] + 0.7 * torch.randn((n, D), device=DEV, generator=gen))
        _fill(db, g, blk)
        src = torch.randperm(n_db, device=DEV, generator=g)[:n_q]
        return db, _unit(db[src] + 0.5 * torch.randn((n_q, D), device=DEV, generator=g) / D ** 0.5)
    _fill(db, g, lambda n, gen: _unit(torch.randn((n, D), device=DEV, generator=gen)))
    q = _unit(torch.randn((n_q, D), device=DEV, generator=g))
    if dist == "straddle":
        target = torch.cat([0.9 + torch.linspace(-5e-5, 5e-5, 400, device=DEV, dtype=torch.float64),
                            torch.full((100,), 0.895, device=DEV, dtype=torch.float64)])
        c = (1.0 / target ** 2 - 1.0).sqrt()
        pos = torch.randperm(n_db, device=DEV, generator=g)[:n_q * 500].view(n_q, 500)
        for j in range(n_q):                          # (q + c n) / sqrt(1 + c^2) with n a unit vector orthogonal to q
            nz = torch.randn((500, D), device=DEV, generator=g).double()
            qj = q[j].double()
            nz = _unit(nz - (nz @ qj)[:, None] * qj[None, :])
            db[pos[j]] = ((qj[None, :] + c[:, None] * nz) / (1.0 + c[:, None] ** 2).sqrt()).float()
    if dist == "near_dup":
        pos = torch.randperm(n_db, device=DEV, generator=g)[:n_q * dup_per_query].view(n_q, dup_per_query)
        for j in range(n_q):
            nz = torch.randn((dup_per_query, D), device=DEV, generator=g)
            nz = nz - (nz @ q[j])[:, None] * q[j][None, :]
            db[pos[j]] = _unit(q[j][None, :] + 0.484 * nz / D ** 0.5)
    return db, q


def independent_ranking(m, index, db, q, k_ext):
    """(idx (nq, k_ext), fp64 scores) by dense 3xTF32 scores -> exact select -> fp64 re-scoring, (score desc, idx asc)."""
    dense = index.scores(q, precision="fp32")
    idx, _ = m.topk_from_scores(dense.t().contiguous(), k_ext + 48)
    del dense
    idx = idx.t().contiguous()
    v64 = (db[idx.reshape(-1)].double().view(idx.shape[0], idx.shape[1], -1) * q.double()[:, None, :]).sum(-1)
    v64, idx = v64.cpu().numpy(), idx.cpu().numpy()
    order = np.lexsort((idx, -v64), axis=1)
    return np.take_along_axis(idx, order, 1)[:, :k_ext], np.take_along_axis(v64, order, 1)[:, :k_ext]


def assert_exact(got_i, got_s, ref_i, ref_v, tol=2e-6):
    """Scores equal to tol position by position; an index mismatch only as a swap inside a reference gap <= tol."""
    k = got_i.shape[1]
    assert np.abs(got_s - ref_v[:, :k]).max() <= tol
    for j in range(got_i.shape[0]):
        for r in np.nonzero(got_i[j] != ref_i[j, :k])[0]:
            assert got_i[j, r] in ref_i[j][np.abs(ref_v[j] - ref_v[j, r]) <= tol], (j, r)


def finalize_both(index, q):
    """One int8 first pass, then the two-tier and the three-tier finalize on its output.
    -> {tiered: (scores, ids, status) numpy}, the shortlist S of every query (a set of slots)."""
    from mdir_b200.search import default_shortlist
    nq, kth = q.shape[0], default_shortlist(K)
    assert index._i8_route(kth, nq)
    route = index._route(kth, nq)
    q8, q_eps = index._pack_q_i8(q)
    tau, cand, cnt, caps = index._first_pass(route, q8, kth, nq)
    out = {}
    for tiered in (False, True):
        s = torch.empty((nq, K), dtype=torch.float32, device=DEV)
        i = torch.empty((nq, K), dtype=torch.int32, device=DEV)
        st = torch.empty((nq,), dtype=torch.int32, device=DEV)
        index.tiered = tiered
        index._finalize(cand, cnt, nq, kth, s, i, None, tau.clone(), st, (q, K), caps, q_eps)
        out[tiered] = (s.cpu().numpy(), i.cpu().numpy(), st.cpu().numpy())
    index.tiered = True
    # S = the kth best candidates by int8 key (the finalize's shortlist); the scan writes rows of cap0 + 148 cap_l keys
    cap0, cap_l = caps
    cand_row = cap0 + 148 * cap_l
    cand, cnt = cand.reshape(-1).cpu().numpy().view(np.uint64), cnt.cpu().numpy()
    shortlists = []
    for j in range(nq):
        row = cand[j * cand_row:(j + 1) * cand_row]
        keys = [row[(0 if sg == 0 else cap0 + (sg - 1) * cap_l):][:min(int(cnt[j, sg]), cap0 if sg == 0 else cap_l)]
                for sg in range(cnt.shape[1])]
        keys = np.sort(np.concatenate(keys))[:kth]
        slots = (keys & np.uint64(0xffffffff)).astype(np.int64) - index.idx_base
        assert keys.size == kth and (slots >= 0).all() and (slots < index.n).all()
        shortlists.append(set(slots.tolist()))
    return out, shortlists


@pytest.fixture(scope="module", params=["randn", "clusters", "near_dup", "straddle"])
def r1m(request, m):
    db, q = build_case(request.param, N_R1M, D_R1M, NQ, {"randn": 61, "clusters": 62, "near_dup": 63, "straddle": 64}[request.param])
    index = m.Index(db, device=DEV)
    yield request.param, db, q, index
    del index, db
    torch.cuda.empty_cache()


def test_tiered_equals_two_tier_and_exact(m, r1m):
    dist, db, q, index = r1m
    out, shortlists = finalize_both(index, q)
    (s2, i2, st2), (s3, i3, st3) = out[False], out[True]
    assert np.array_equal(i2, i3) and np.array_equal(s2.view(np.uint32), s3.view(np.uint32)) and np.array_equal(st2, st3)
    ok = st3 == 0
    assert ok.all() if dist == "randn" else ok.any(), st3      # bench.py's kind of data: every query certified
    ref_i, ref_v = independent_ranking(m, index, db, q, K + 16)
    assert_exact(i3[ok], s3[ok].astype(np.float64), ref_i[ok], ref_v[ok])
    # the public route agrees (a flagged block is redone through the bf16 route)
    s, i = index.search(q, K, precision="fp32")
    assert np.array_equal(i.cpu().numpy()[ok], i3[ok]) and np.array_equal(s.cpu().numpy()[ok], s3[ok])
    from_f = sum(len(set(i3[j].tolist()) - shortlists[j]) for j in range(NQ))
    print("tiered %s: identical to two tiers; %d of %d certified; %d emitted rows came from F" % (dist, ok.sum(), NQ, from_f))
    if dist == "straddle":
        # the int8 shortlist holds about a third of the 400 rows around t0: most of the top-100 must come through F
        assert from_f >= 20 * NQ


def test_tier2_bound_holds_on_measured_scores(m):
    """max over rows of |s16 - fp32| / eps16 < 1, s16 = the bf16-rounded row against the fp32 query in fp32."""
    worst = 0.0
    for dist, seed in (("randn", 71), ("clusters", 72), ("near_dup", 73)):
        db, q = build_case(dist, 200000, 2048, 16, seed, dup_per_query=100)
        index = m.Index(db, device=DEV)
        st = index.stats().double().cpu().numpy()
        s32 = q @ db.t()
        s16 = q @ index.db16.float().t()
        qn = q.double().norm(dim=1).cpu().numpy()
        acc = 1.25 * 2048 * 2.0 ** -24
        eps16 = (np.sqrt(st[0]) * qn + acc * (np.sqrt(st[1]) + np.sqrt(st[0])) * qn + acc * np.sqrt(st[1]) * qn) * 1.001 + 1e-7
        ratio = float(((s16 - s32).abs().max(dim=1).values.double().cpu().numpy() / eps16).max())
        print("tier-2 bound %s: max |s16 - fp32| / eps16 = %.3f (eps16 %.2e)" % (dist, ratio, eps16.max()))
        worst = max(worst, ratio)
        del index, db, s32, s16
    assert 0.0 < worst < 1.0


@pytest.mark.parametrize("k", [40, 100])
def test_search_scores_equal_range_search_scores(m, k):
    """Every fp32 re-score uses one summation order, whether its row was paired or not: a row's search score is its
    range_search score bit for bit, at k = 40 (64-row shortlist) as at k = 100."""
    db, q = build_case("randn", 60000, 2048, 70, 81)
    db[:70] = _unit(q + 0.3 * torch.randn(q.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(5)) / 2048 ** 0.5)
    index = m.Index(db, device=DEV)
    s, i = index.search(q, k, precision="fp32")
    s, i = s.cpu().numpy(), i.cpu().numpy()
    lims, rs, ri = index.range_search(q, torch.from_numpy(s[:, k - 1].copy()))
    lims, rs, ri = lims.cpu().numpy(), rs.cpu().numpy(), ri.cpu().numpy()
    for j in range(q.shape[0]):
        got = dict(zip(ri[lims[j]:lims[j + 1]].tolist(), rs[lims[j]:lims[j + 1]].view(np.uint32).tolist()))
        assert all(got.get(int(a)) == int(b) for a, b in zip(i[j], s[j].view(np.uint32))), j
