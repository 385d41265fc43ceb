"""The Lw projection y = P[:dims] (v - m) (optionally y / (||y|| + eps)) against fp64, at the production width.

Every route is judged by one condition-scaled measure.  For entry j of a descriptor,

    e_j = max(0, |got_j - ref_j| - RENORM_ULPS * 2^-24 * |ref_j|) / c_j,    c_j = sum_i |P_ji x_i|

with x = v - m formed in fp32 (as the kernels and the reference's fp32 wrapper do) and everything else in fp64.  When the
output is renormalised, c_j is divided by ||y|| + eps as well, and the RENORM_ULPS term allows for the fp32 norm, its square
root, the reciprocal and the final product: a relative error of the scale factor, so a few ulps of ref_j.  Without
renormalisation that term is zero.  An fp32 dot product's error scales with c_j, so the same bar holds for a
well-conditioned random P and an ill-conditioned learned one, and an entry that happens to be near zero is not judged
against its own tiny magnitude.  The bar is BAR = 2e-6, the fp32-faithful figure of DESIGN.md section 2.1.

Routes: the tensor-core projection (3xTF32 split on sim_scan_kernel<TF32>, split-K partial planes, one or two streams),
the chained fp32 scan of Index.scores / ranks as the calibration point, the CUDA-core GEMV / SGEMM projection, the batched
head at the C2 shape (192 images x 3 scales x 2048 channels), its CUDA-graph capture and whitenapply.  Each check prints
its measured max e (run with -s to see them).
"""
import ctypes
import functools

import numpy as np
import pytest
import torch

from oracle import oracle

pytestmark = pytest.mark.gpu

DEV = "cuda"
BAR = 2e-6
RENORM_ULPS = 8
U32 = 2.0 ** -24
EPS = 1e-6


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    from mdir_b200 import _lib
    _lib.check(_lib.lib().mdir_device_check(), "device check")
    return mdir_b200


# ------------------------------------------------------------------ inputs (seeded, numpy fp32)
def _unit_rows(n, D, seed, kind):
    """kind "nonneg": non-negative unit rows (GeM of ReLU maps); "signed": signed unit rows."""
    x = np.random.default_rng(seed).standard_normal((n, D))
    if kind == "nonneg":
        x = np.abs(x)
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


def _mean(v, seed, kind):
    """kind "bench": 0.01 randn (bench.py's m); "data": the actual mean of the rows."""
    if kind == "bench":
        return (0.01 * np.random.default_rng(seed).standard_normal(v.shape[1])).astype(np.float32)
    return v.astype(np.float64).mean(axis=0).astype(np.float32)


@functools.lru_cache(maxsize=None)
def _lw_P(kind, D):
    """(D, D) fp32.  "randn": bench.py's randn / sqrt(C).  "learned": diag(s) Q with Q orthogonal (QR of a seeded randn)
    and s log-spaced over 1 ... 1e3 -- the eig^-1/2 scaling of a learned Lw makes it ill-conditioned."""
    rng = np.random.default_rng(1000 + D)
    if kind == "randn":
        return (rng.standard_normal((D, D)) / np.sqrt(D)).astype(np.float32)
    q, r = np.linalg.qr(rng.standard_normal((D, D)))
    q *= np.sign(np.diag(r))[None, :]
    return (np.logspace(0.0, 3.0, D)[:, None] * q).astype(np.float32)


# (P kind, v kind, m kind); each tensor-core case runs two of them, so every shape sees all four over the n grid
COMBOS = [("randn", "nonneg", "bench"), ("learned", "nonneg", "data"), ("randn", "signed", "data"), ("learned", "signed", "bench")]


def _inputs(n, D, combo, seed):
    pk, vk, mk = combo
    v = _unit_rows(n, D, seed, vk)
    return v, _mean(v, seed + 1, mk), _lw_P(pk, D)


# ------------------------------------------------------------------ reference and error measure
def _reference(v, mm, P, dims):
    """fp64 y = P[:dims] (v - m) with x = v - m in fp32, and the condition c = |P[:dims]| |x|: (n, dims) each."""
    x = (v - mm[None, :]).astype(np.float64) if mm is not None else v.astype(np.float64)
    Pd = P[:dims].astype(np.float64)
    return x @ Pd.T, np.abs(x) @ np.abs(Pd).T


def _max_e(got, y, c, renorm, eps=EPS):
    """max_j e_j (see the module docstring); got (n, dims) from the device, y / c from _reference."""
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    got = got.astype(np.float64)
    if renorm:
        nrm = np.sqrt((y * y).sum(axis=1, keepdims=True)) + eps
        ref, cond = y / nrm, c / nrm
        d = np.maximum(np.abs(got - ref) - RENORM_ULPS * U32 * np.abs(ref), 0.0)
    else:
        ref, cond, d = y, c, np.abs(got - y)
    assert np.all(np.isfinite(got))
    return float((d / np.maximum(cond, np.finfo(np.float64).tiny)).max())


def _check(tag, got, y, c, renorm, eps=EPS):
    e = _max_e(got, y, c, renorm, eps)
    print("max_e %-58s %.3e" % (tag, e))
    assert e <= BAR, (tag, e)
    return e


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


# ------------------------------------------------------------------ 1. tensor-core projection (3xTF32, split-K)
# (D, dims): the k_split / k-blocks-per-split rows of whiten_plan -- 12 x 1 at 128, 24 x 2 at 512, 32 x 6 at
# 2048 -> 512, 18 x 11 (<= 128 descriptors) and 9 x 22 (more) at 2048 -> 2048; dims 250 and 100 take the unfused
# epilogue (sum_partials_kernel + row_l2n_kernel) or a ragged 256-row tile.
TC_SHAPES = [(2048, 2048), (2048, 512), (2048, 250), (2048, 100), (512, 512), (128, 128)]
# 5: one block; 128: one full block; 129: 80 + 49 on two streams; 192: 96 + 96; 600: 4 x 128 + 88, odd block count
TC_NS = [5, 128, 129, 192, 600]


@pytest.mark.parametrize("D,dims", TC_SHAPES)
@pytest.mark.parametrize("n", TC_NS)
def test_tensor_core_projection_vs_fp64(m, n, D, dims):
    from mdir_b200 import wrappers
    for combo in COMBOS[(TC_NS.index(n) % 2) * 2:][:2]:
        v, mm, P = _inputs(n, D, combo, 10 * n + D)
        y, c = _reference(v, mm, P, dims)
        Pd = _dev(P)
        Px3 = wrappers.split_lw(Pd)
        for renorm in (True, False):
            got = wrappers.whiten_project(_dev(v), _dev(mm), Pd, dims, renorm_eps=EPS if renorm else -1.0, Px3=Px3)
            _check("tc n=%d D=%d dims=%d P=%s v=%s m=%s renorm=%d" % ((n, D, dims) + combo + (renorm,)), got, y, c, renorm)


# ------------------------------------------------------------------ 2. the chained fp32 scan: same split, <= 16 MMAs per accumulation
@pytest.mark.parametrize("dims", [2048, 512, 250])
@pytest.mark.parametrize("n", [70, 128, 600])
def test_chained_fp32_scores_at_2048(m, n, dims):
    """Index(P[:dims]).scores(x, "fp32") computes hi.hi + hi.lo + lo.hi like the projection, chained in 48 chunks of
    4 k-blocks at D = 2048; query blocks wider than kChainMaxN = 96 go as two launches (n = 128, 600)."""
    D = 2048
    for combo in COMBOS[:2]:
        v, mm, P = _inputs(n, D, combo, 7 * n + dims)
        y, c = _reference(v, mm, P, dims)
        x = (v - mm[None, :]).astype(np.float32)
        index = m.Index(P[:dims], device=DEV, keep_fp32=True)
        _check("chained n=%d D=%d dims=%d P=%s v=%s m=%s" % ((n, D, dims) + combo), index.scores(x, precision="fp32"), y, c, False)


def _assert_same_order(got, sc, tol):
    """got (n_db, nq) full ranking vs fp64 scores sc (n_db, nq): got must be a permutation of the rows, and the row it
    puts at position r must score, in fp64, within `tol` of the r-th best fp64 score -- rows may only trade places with
    rows that tie with them to within summation-order noise."""
    n_db, nq = got.shape
    assert np.array_equal(np.sort(got, axis=0), np.broadcast_to(np.arange(n_db)[:, None], got.shape))
    ref_sorted = -np.sort(-sc, axis=0)
    gap = np.abs(np.take_along_axis(sc, got, axis=0) - ref_sorted)
    r, j = np.unravel_index(int(gap.argmax()), gap.shape)
    assert gap[r, j] <= tol, (r, j, got[r, j], gap[r, j])


@pytest.mark.parametrize("n_q", [70, 96, 97, 200])
def test_chained_fp32_ranks_at_2048(m, n_q):
    """A plain fp32 search of unit 2048-D descriptors: 20,000 x 2048, queries on both sides of kChainMaxN = 96.
    |score| <= c <= 1 for unit rows, so twice the bar is an absolute 2 * BAR on the scores."""
    db = _unit_rows(20000, 2048, 31, "signed")
    q = _unit_rows(n_q, 2048, 32 + n_q, "signed")
    index = m.Index(db, device=DEV, keep_fp32=True)
    y, c = _reference(q, None, db, 20000)                          # (n_q, n_db)
    _check("chained scores n_q=%d n_db=20000 D=2048" % n_q, index.scores(q, precision="fp32"), y, c, False)
    ranks = index.ranks(q, precision="fp32").cpu().numpy()
    _assert_same_order(ranks, np.ascontiguousarray(y.T), 2 * BAR)


# ------------------------------------------------------------------ 3. CUDA-core projection (GEMV, SGEMM<32>, SGEMM<64>, scalar loads)
@pytest.mark.parametrize("n,D,dims", [(1, 2048, 2048), (2, 2048, 2048), (3, 2048, 512), (4, 2048, 250),
                                      (5, 2048, 2048), (600, 2048, 2048),
                                      (2, 2046, 2046), (5, 2046, 2046), (600, 2046, 2046)])
def test_cuda_core_projection_vs_fp64(m, n, D, dims):
    """n <= 4: whiten_gemv_kernel<n>; more: whiten_sgemm_kernel<32>, or <64> once ceil(dims/64) ceil(n/64) >= 296
    (600 x 2048); D = 2046: the scalar loads (the tensor-core route needs D % 4 == 0)."""
    from mdir_b200 import wrappers
    for combo in COMBOS[(n % 2) * 2:][:2]:
        v, mm, P = _inputs(n, D, combo, 13 * n + D)
        y, c = _reference(v, mm, P, dims)
        Pd = _dev(P)
        for renorm in (True, False):
            got = wrappers.whiten_project(_dev(v), _dev(mm), Pd, dims, renorm_eps=EPS if renorm else -1.0, Px3=None)
            _check("cuda-core n=%d D=%d dims=%d P=%s v=%s m=%s renorm=%d" % ((n, D, dims) + combo + (renorm,)), got, y, c, renorm)


# ------------------------------------------------------------------ 4./5. the batched head at the C2 shape
HWS = [(32, 24), (23, 17), (16, 12)]
C2 = 2048
P_GEM = 2.9137


def _maps(n_img, hws, seed):
    """bench.py's head inputs: n_img x len(hws) maps of randn(1, C, h, w).clamp(min=0), image-major."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    fm = [torch.randn((1, C2, h, w), device=DEV, generator=g).clamp_(min=0) for _ in range(n_img) for (h, w) in hws]
    return fm, g


@pytest.fixture(scope="module")
def c2(m):
    """192 images x 3 scales x 2048 channels seeded as in bench.py, with its P (kind a) and m."""
    fm, g = _maps(192, HWS, 7)
    P = torch.randn((C2, C2), device=DEV, generator=g) / C2 ** 0.5
    mm = torch.randn((C2, 1), device=DEV, generator=g) * 0.01
    return fm, P.cpu().numpy(), mm.cpu().numpy().reshape(-1)


def _lw_kinds(c2):
    _, P_bench, m_bench = c2
    return [("randn", P_bench), ("learned", _lw_P("learned", C2))], m_bench


def test_head_c2_projection_vs_fp64(m, c2):
    """RetrievalHead with and without Lw on the same packed maps: the unwhitened output is exactly the v the projection
    receives, so the whitened one is judged against fp64 P (v - m) of it -- the projection alone, at production size."""
    fm = c2[0]
    plain = m.RetrievalHead("gem", p=P_GEM, nscales=3, device=DEV)
    packed = plain.pack(fm)
    v = plain(packed).cpu().numpy()
    assert v.shape == (192, C2)
    kinds, mm = _lw_kinds(c2)
    for name, P in kinds:
        head = m.RetrievalHead("gem", p=P_GEM, whitening={"P": P, "m": mm}, nscales=3, device=DEV)
        y, c = _reference(v, mm, P, C2)
        _check("head C2 192 x 3 x 2048 P=%s" % name, head(packed), y, c, True)


def test_head_c2_vs_oracle_and_composite(m, c2):
    """End to end against oracle.gem_head on the images at the ends and on both sides of the 96 + 96 block boundary;
    the mdir_gem_head composite equals RetrievalHead bit for bit at this shape."""
    from mdir_b200 import _lib
    fm = c2[0]
    kinds, mm = _lw_kinds(c2)
    lib = _lib.lib()
    for name, P in kinds + [("none", None)]:
        lw = None if P is None else {"P": P, "m": mm}
        head = m.RetrievalHead("gem", p=P_GEM, whitening=lw, nscales=3, device=DEV)
        pm = head.pack(fm)
        out = head(pm)
        for i in (0, 95, 96, 191):
            per = [fm[3 * i + s].cpu().numpy() for s in range(3)]
            ref = oracle.gem_head(per, P_GEM, 1e-6, mm if P is not None else None, P)
            np.testing.assert_allclose(out[i].cpu().numpy().astype(np.float64), ref.astype(np.float64), rtol=2e-5, atol=3e-7,
                                       err_msg="P=%s image %d" % (name, i))
        dims = C2 if P is not None else 0
        comp = torch.empty((192, C2), dtype=torch.float32, device=DEV)
        ws = torch.empty((lib.mdir_gem_head_workspace_bytes(192, 3, C2, dims),), dtype=torch.uint8, device=DEV)
        with torch.cuda.device(out.device):
            _lib.check(lib.mdir_gem_head(0, ctypes.c_void_p(pm.base), _lib.ptr(pm.off), _lib.ptr(pm.hw), 192, 3, C2, 0, P_GEM, 1e-6, head.msp,
                                         _lib.ptr(head.m) if P is not None else None, _lib.ptr(head.P) if P is not None else None,
                                         _lib.ptr(head.Px3) if P is not None else None, dims, _lib.ptr(comp), _lib.ptr(ws), _lib.stream()),
                       "mdir_gem_head")
        assert torch.equal(comp, out), name


@pytest.mark.parametrize("n_img", [192, 600])
def test_captured_head_two_streams(m, c2, n_img):
    """head.capture(): the two-stream fork / join recorded into a CUDA graph.  192 = 96 + 96 (one block per stream);
    600 = 4 x 128 + 88 (odd block count: three blocks on the caller's stream, two on the side stream).  The replay equals
    the eager head bit for bit and follows maps mutated in place, in blocks of both streams."""
    if n_img == 192:
        fm = c2[0]
    else:
        fm, _ = _maps(n_img, [(16, 12), (11, 8), (8, 6)], 11)       # smaller maps: the projection is what is under test
    _, P_bench, m_bench = c2
    head = m.RetrievalHead("gem", p=P_GEM, whitening={"P": P_bench, "m": m_bench}, nscales=3, device=DEV)
    packed = head.pack(fm)
    replay = head.capture(packed)
    eager = head(packed).clone()
    assert torch.equal(replay(), eager)
    rows = 96 if n_img == 192 else 128                                  # descriptors per projection block
    mutated = (0, rows + 2, n_img - 1)                                  # block 0 (caller's stream), block 1 (side stream), the last block
    for i in mutated:
        fm[3 * i + 1][:, :C2 // 2].mul_(0.5)                           # same storage, new contents (and a new direction: the
    now = replay().clone()                                             # per-scale L2N would cancel a uniform scale)
    assert torch.equal(now, head(packed))
    keep = torch.ones(n_img, dtype=torch.bool, device=DEV)
    keep[list(mutated)] = False
    assert torch.equal(now[keep], eager[keep])
    for i in mutated:
        assert not torch.equal(now[i], eager[i]), i
        fm[3 * i + 1][:, :C2 // 2].mul_(2.0)
    assert torch.equal(replay(), eager)


# ------------------------------------------------------------------ 6. whitenapply over a database
@pytest.mark.parametrize("P_kind", ["randn", "learned"])
def test_whitenapply_2048_vs_oracle(m, P_kind):
    """cirtorch's whitenapply on a (2048, 1000) fp64 matrix (8 blocks of <= 128 on two streams), judged against
    oracle.whitenapply.  The inputs are fp32 values held in fp64, so the oracle is the exact result of what the device is
    given; the device's fp32 centring adds at most one rounding of x, u c_j, to the error."""
    D, N = 2048, 1000
    X = _unit_rows(N, D, 41, "nonneg").T.astype(np.float64)
    mm = X.mean(axis=1, keepdims=True).astype(np.float32).astype(np.float64)
    P = _lw_P(P_kind, D).astype(np.float64)
    for dims in (None, 512):
        out = m.whitenapply(X, mm, P, dims)
        ref = oracle.whitenapply(X, mm, P, dims)
        assert out.dtype == np.float64 and out.shape == ref.shape
        y, c = _reference(X.T, mm.reshape(-1), P, dims or D)          # fp64 centring: y is the oracle's before the norm
        np.testing.assert_allclose(y / (np.linalg.norm(y, axis=1, keepdims=True) + EPS), ref.T, rtol=1e-12, atol=1e-15)
        _check("whitenapply 2048 x 1000 P=%s dims=%s" % (P_kind, dims), out.T, y, c, True)
