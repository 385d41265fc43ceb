"""The fused int8 scan (sim_scan_kernel<kKindI8>) rotates its accumulators per 128-row half through three TMEM
buffers (two beyond 80 queries).  Each half has its own rows, row scales, live word and buffer, and its s32 sums are
exact, so every CTA's candidate list must equal an independent reconstruction exactly: torch._int_mm accumulators of
db8 against both query planes, through the epilogue's fp32 formula, filtered by the published thresholds and assigned
to the CTA that owns each tile.  Only rows whose score lies within one ulp of the threshold may differ (fp32 rounding
of the reconstruction's fused multiply-add); they are listed.

The shapes give CTAs odd and even tile counts (so the buffer rotation wraps at different halves), a last tile whose
second half lies wholly past the end, an extent below capacity, 10 % of the rows removed, 16 queries and 96 queries
(two buffers).  A half scored with another half's row scale, live word or buffer changes rows far from the threshold."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TILE = 256
KTH = 128


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    return mdir_b200


def _balanced_grid(n_work, max_ctas):
    """common.cuh:balanced_grid."""
    if n_work <= max_ctas:
        return n_work
    rounds = -(-n_work // max_ctas)
    return -(-n_work // rounds)


def _cta_tiles(n_db, n_end, sms):
    """Tiles whose rows each CTA of a FUSED launch counts: launch_scan's grid and make_span / next_item's work list."""
    n_tiles = -(-n_db // TILE)
    g = _balanced_grid(n_tiles, min(sms, 148, n_tiles // 2))
    stride, n_sample, n_work = n_tiles // g, g, n_tiles - g
    sample = [c * stride for c in range(g)]
    if n_end < n_db:
        t_used = -(-n_end // TILE)
        stride = max(1, t_used // g)
        n_sample = min(g, -(-t_used // stride))
        sample = [c * stride if c < n_sample else -1 for c in range(g)]
        n_work = t_used - n_sample

    def tile_of_work(j):
        per = stride - 1
        in_groups = n_sample * per
        if j < in_groups:
            grp = j // per
            return grp * stride + 1 + (j - grp * per)
        return n_sample * stride + (j - in_groups)

    return [([sample[c]] if sample[c] >= 0 else []) + [tile_of_work(j) for j in range(c, n_work, g)] for c in range(g)]


def _key_scores(keys):
    o = ~(keys >> np.uint64(32)).astype(np.uint32)
    u = np.where(o >> np.uint32(31) != 0, o ^ np.uint32(0x80000000), o ^ np.uint32(0xffffffff)).astype(np.uint32)
    return u.view(np.float32)


@pytest.mark.parametrize("n_rows,cap,nq,D,removed", [
    (114700, None, 70, 256, 0.0),       # last tile: 12 rows, its second half wholly past the end
    (100037, None, 70, 512, 0.1),       # 3 or 2 tiles per CTA
    (100037, 160000, 61, 256, 0.1),     # extent below capacity
    (50301, None, 16, 256, 0.0),        # 16 queries
    (70001, None, 96, 256, 0.1),        # 96 queries: two accumulator buffers
])
def test_int8_fused_candidates_equal_reconstruction(m, monkeypatch, n_rows, cap, nq, D, removed):
    S, lib, _lib = m.search, m.lib(), m._lib
    monkeypatch.setattr(S, "I8_MIN_ROWS", 0)
    g = torch.Generator(device=DEV).manual_seed(n_rows + nq)
    db = torch.randn((n_rows, D), device=DEV, generator=g)
    db /= db.norm(dim=1, keepdim=True)
    q32 = torch.randn((nq, D), device=DEV, generator=g)
    q32 /= q32.norm(dim=1, keepdim=True)
    index = m.Index(db, device=DEV, capacity=cap)
    rng = np.random.default_rng(n_rows)
    if removed:
        index.remove(rng.choice(n_rows, int(removed * n_rows), replace=False))
    index.stats()
    assert index.db8 is not None
    (q8, qsc), _ = index._pack_q_i8(q32)
    tau, cand, cnt = index._cand_bufs(nq)
    _lib.check(lib.mdir_sim_scan_fused_i8_extent(_lib.ptr(index.db8), _lib.ptr(index.row_scale), index.n, _lib.ptr(q8), _lib.ptr(qsc), nq, D,
                                                 KTH, _lib.ptr(tau), index.idx_base, _lib.ptr(cand), _lib.ptr(cnt), 0, S.FUSED_CAP_L,
                                                 _lib.ptr(index._fused_ws()), _lib.ptr(index.live), _lib.ptr(index.n_scan), _lib.stream()),
               "mdir_sim_scan_fused_i8_extent")
    # ---- reconstruction: exact s32 sums, then fmul(fmaf(hi, s_hi, fmul(lo, s_lo)), s_r) in fp32 (the fma in fp64:
    # the product is exact there, so only the final rounding to fp32 can differ, by one ulp at a halfway case)
    n_pad = q8.shape[0] // 2
    acc_hi = torch._int_mm(index.db8, q8[:n_pad].t())[:, :nq]
    acc_lo = torch._int_mm(index.db8, q8[n_pad:].t())[:, :nq]
    t_lo = acc_lo.float() * qsc[:, 1]
    s = (acc_hi.float().double() * qsc[:, 0].double() + t_lo.double()).float() * index.row_scale[:, None]
    torch.cuda.synchronize()
    s = s.cpu().numpy()
    n_end = n_rows
    live = index._live_host.copy()
    live[n_end:] = False
    tau_k = tau[:nq].cpu().numpy().view(np.uint64)
    assert (tau_k != 0).all(), "threshold exchange timed out"
    assert ((tau_k & np.uint64(0xffffffff)) == np.uint64(0xffffffff)).all()
    tau_f = _key_scores(tau_k)
    counts = cnt[:nq].cpu().numpy().view(np.uint32).astype(np.int64)
    assert counts[:, 0].max() == 0
    row_len = 148 * S.FUSED_CAP_L
    flat = cand.view(-1)[:nq * row_len].cpu().numpy().view(np.uint64).reshape(nq, row_len)
    per_cta = _cta_tiles(index.n, n_end, torch.cuda.get_device_properties(DEV).multi_processor_count)
    assert counts[:, 1 + len(per_cta):].max(initial=0) == 0
    near_all, compared = [], 0
    for j in range(nq):
        keys = S.make_keys_host(s[:, j], np.arange(index.n) + index.idx_base)
        ok = live & (keys <= tau_k[j]) & (s[:, j] >= tau_f[j])
        near = np.abs(s[:, j].astype(np.float64) - float(tau_f[j])) <= float(np.spacing(np.float32(abs(tau_f[j]))))
        for c, tiles in enumerate(per_cta):
            rows = np.concatenate([np.arange(t * TILE, (t + 1) * TILE) for t in tiles]) if tiles else np.zeros(0, np.int64)
            rows = rows[rows < index.n]
            want = keys[rows[ok[rows]]]
            assert counts[j, 1 + c] <= S.FUSED_CAP_L, "candidate segment overflowed"
            got = flat[j, c * S.FUSED_CAP_L:c * S.FUSED_CAP_L + counts[j, 1 + c]]
            assert len(np.unique(got)) == len(got)
            diff = np.setxor1d(got, want)
            drows = (diff & np.uint64(0xffffffff)).astype(np.int64) - index.idx_base
            assert np.all(near[drows]), (j, c, drows[~near[drows]][:8])
            near_all += [(j, int(r)) for r in drows]
            compared += len(want)
    assert compared > nq * KTH
    if near_all:
        print("rows within one ulp of the threshold that differ (query, row):", near_all)
