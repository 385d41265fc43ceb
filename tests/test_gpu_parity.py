"""GPU parity tests: the CUDA path (through the C ABI) against oracle/ and the committed
golden vectors (outputs of the reference itself), on the same seeded inputs.

Bars (BASELINE.json north_star): CLAHE and sort/top-k indexing bit-exact; pooled / whitened
descriptors within 1e-5 relative; similarity scores within 2e-3 absolute on the bf16 path;
mAP within 0.01."""
import os
import types

import numpy as np
import pytest
import torch

from oracle import oracle, synth

pytestmark = pytest.mark.gpu

DEV = "cuda"
REL = 1e-5


def close(a, b, rtol=REL, atol=0.0):
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    np.testing.assert_allclose(np.asarray(a, np.float64), np.asarray(b, np.float64), rtol=rtol, atol=atol)


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


@pytest.fixture(scope="module")
def m():
    import mdir_b200
    from mdir_b200 import _lib
    _lib.check(_lib.lib().mdir_device_check(), "device check")
    return mdir_b200


# ------------------------------------------------------------------ pooling / L2N
@pytest.mark.parametrize("si", range(len(synth.POOL_SHAPES)))
@pytest.mark.parametrize("kind", ["relu", "signed", "zeros"])
def test_pooling_vs_oracle_and_golden(m, golden, si, kind):
    g = golden("pooling")
    x = synth.fmap(synth.POOL_SHAPES[si], 100 + si, kind)
    xd = dev(x)
    tag = "s%d_%s" % (si, kind)
    assert np.array_equal(m.MAC()(xd).cpu().numpy(), g[tag + "_mac"])              # max is exact
    close(m.SPoC()(xd), g[tag + "_spoc"], atol=1e-7)
    close(m.SPoC()(xd), oracle.spoc(x), atol=1e-7)
    close(m.L2N()(m.MAC()(xd)), g[tag + "_l2n_mac"], atol=1e-7)
    for p in synth.POOL_PS:
        out = m.GeM(p=p).to(DEV)(xd)
        assert out.shape == (x.shape[0], x.shape[1], 1, 1)
        close(out, oracle.gem(x, p))
        close(out, g[tag + "_gem_p%g" % p])
        close(m.L2N()(out), g[tag + "_l2n_gem_p%g" % p], atol=1e-8)


def test_gem_zero_and_learned_p(m):
    z = torch.zeros(1, 8, 5, 5, device=DEV)
    close(m.gem(z, 3.0), np.full((1, 8, 1, 1), 9.99999656e-07), rtol=1e-6)
    gm = m.GeM(p=3).to(DEV)
    gm.p.data.fill_(2.5)                       # learnable parameter is honoured
    x = synth.fmap((1, 16, 9, 7), 5)
    close(gm(dev(x)), oracle.gem(x, 2.5))
    assert "p=2.5000" in repr(gm)


def test_l2n_inner(m):
    x = synth.fmap((3, 37, 5, 4), 9, "signed")
    close(m.l2n(dev(x)), oracle.l2n(x), atol=1e-8)


def test_pool_full_size_properties(m):
    # C1/C2 shapes: (B,2048,32,24) maps; size-independent properties instead of a CPU oracle
    g = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randn((24, 2048, 32, 24), device=DEV, generator=g).clamp_(min=0)
    p = 2.9137
    y = m.gem(x, p)
    mx, mean = m.mac(x), m.spoc(x)
    assert torch.all(y <= mx * (1 + 1e-5) + 1e-6) and torch.all(y + 1e-6 >= mean * (1 - 1e-5))     # power-mean inequality
    close(m.gem(x * 2.0, p), (y * 2.0).cpu().numpy(), rtol=2e-5)                               # homogeneity
    sub = x[5:6, 100:164].contiguous()
    close(m.gem(sub, p), oracle.gem(sub.cpu().numpy(), p))
    close(y[5:6, 100:164], oracle.gem(sub.cpu().numpy(), p))


# ------------------------------------------------------------------ head
def _fake_model(pooling, p):
    return types.SimpleNamespace(meta={"pooling": pooling, "regional": False, "whitening": False, "out_channels": 128},
                                 pool=types.SimpleNamespace(p=torch.tensor([p])))


def test_head_vs_golden(m, golden):
    g = golden("head")
    C = 128
    hw = [(32, 24), (23, 17), (16, 12)]
    lw = {"m": g["lw_m"], "P": g["lw_P"]}
    for pooling, ps in (("gem", (3.0, 2.9137)), ("mac", (3.0,)), ("spoc", (3.0,))):
        for p in ps:
            pool = {"gem": lambda: m.GeM(p=p), "mac": m.MAC, "spoc": m.SPoC}[pooling]().to(DEV)
            model = _fake_model(pooling, p)
            ms = m.CirMultiscaleAggregation(True, DEV)
            for img in range(3):
                fm = [synth.fmap((1, C, h, w), 200 + 10 * img + s, "relu") for s, (h, w) in enumerate(hw)]
                # the reference's per-scale tail: norm(pool(o)).squeeze().permute  (imageretrievalnet.py:107-115)
                outs = []
                for s in range(3):
                    o = m.L2N()(pool(dev(fm[s]))).squeeze(-1).squeeze(-1).permute(1, 0)
                    close(o, g["tail_%s_p%g_i%d_s%d" % (pooling, p, img, s)], atol=1e-8)
                    outs.append(o)
                v = ms.postprocess([o.clone() for o in outs], model, False)
                close(v, g["agg_%s_p%g_i%d" % (pooling, p, img)], atol=1e-8)
                v1 = m.CirMultiscaleAggregation([1], DEV).postprocess([outs[0].clone()], model, False)
                close(v1, g["agg1_%s_p%g_i%d" % (pooling, p, img)], atol=1e-8)
                for dims in (None, 64, 32):
                    wh = m.CirtorchWhiten(lw, dims, DEV)
                    w = wh.postprocess(v.clone(), model, None)
                    assert w.shape == (dims or C,)
                    close(w, g["wh_%s_p%g_i%d_d%s" % (pooling, p, img, dims)], rtol=2e-5, atol=3e-7)
    out = m.whitenapply(g["whitenapply_X"], g["lw_m"], g["lw_P"])
    assert out.dtype == np.float64 and out.shape == (128, 40)
    close(out, g["whitenapply_full"], rtol=2e-5, atol=3e-7)
    close(m.whitenapply(g["whitenapply_X"], g["lw_m"], g["lw_P"], 48), g["whitenapply_d48"], rtol=2e-5, atol=3e-7)


def test_batched_head_vs_oracle(m, golden):
    g = golden("head")
    C = 128
    lw = {"m": g["lw_m"], "P": g["lw_P"]}
    hws = [[(32, 24), (23, 17), (16, 12)], [(24, 32), (17, 23), (12, 16)], [(31, 21), (22, 15), (16, 11)], [(8, 8), (6, 6), (4, 4)]]
    fmaps, flat = [], []
    for i, hw in enumerate(hws * 3):                      # 12 ragged images (> 4: exercises the SGEMM projection)
        per = [synth.fmap((1, C, h, w), 900 + 7 * i + s, "relu") for s, (h, w) in enumerate(hw)]
        fmaps.append(per)
        flat += [dev(f) for f in per]
    for dims in (None, 64):
        head = m.RetrievalHead("gem", p=2.9137, whitening=lw, dimensions=dims, nscales=3, device=DEV)
        out = head(flat).cpu().numpy()
        for i, per in enumerate(fmaps):
            ref = oracle.gem_head(per, 2.9137, 1e-6, lw["m"], lw["P"], dims)
            close(out[i], ref, rtol=2e-5, atol=3e-7)
    # the head recorded into a CUDA graph over a static arena: replays follow the arena's contents
    head = m.RetrievalHead("gem", p=2.9137, whitening=lw, dimensions=None, nscales=3, device=DEV)
    packed = head.pack(flat)
    replay = head.capture(packed)
    eager = head(packed).clone()
    assert bool((replay() == eager).all())
    flat[0].mul_(0.5)                                     # same storage, new contents
    assert bool((replay() == head(packed)).all()) and not bool((replay()[0] == eager[0]).all())
    flat[0].mul_(2.0)
    # single-scale, no whitening, packed NCHW input (C1 shape family)
    x = synth.fmap((5, C, 32, 24), 77)
    head = m.RetrievalHead("gem", p=3.0, nscales=1, device=DEV)
    out = head(dev(x)).cpu().numpy()
    for i in range(5):
        close(out[i], oracle.gem_head([x[i:i + 1]], 3.0, 1e-6), atol=1e-8)


# ------------------------------------------------------------------ CLAHE
def test_clahe_bit_exact_all_cases(m, golden):
    g = golden("clahe")
    cases = synth.clahe_cases()
    for clip in (4, 2, 40):
        sel = [c for c in cases if c[3] == clip]
        imgs = [synth.image_u8(hw, dist, seed) for (_, hw, dist, _, seed) in sel]
        outs = m.clahe_u8([dev(i) for i in imgs], clip, (8, 8))               # one ragged batch per clip limit
        for (key, hw, dist, _, seed), img, out in zip(sel, imgs, outs):
            o = out.cpu().numpy()
            assert synth.sha(img) == str(g["in_sha_" + key])
            assert synth.sha(o) == str(g["out_sha_" + key]), key
            if hw in synth.CLAHE_SMALL:
                assert np.array_equal(o, g["out_" + key]), key
            if hw in synth.CLAHE_SMALL or dist == "gamma":
                assert np.array_equal(o, oracle.clahe_u8(img, clip, 8, 8)), key


def test_clahe_grid_pitch_and_wrappers(m, golden):
    g = golden("clahe")
    img = synth.image_u8((127, 93), "gamma", 77)
    assert np.array_equal(m.clahe_u8(dev(img), 3, (4, 6)).cpu().numpy(), g["grid4x6_127x93"])
    # strided (pitch != width) view and a (B,H,W) batch
    big = dev(synth.image_u8((127, 200), "uniform", 3))
    view = big[:, 50:143]
    assert np.array_equal(m.clahe_u8(view, 4, (8, 8)).cpu().numpy(), oracle.clahe_u8(view.cpu().numpy(), 4, 8, 8))
    batch = np.stack([synth.image_u8((96, 128), d, 40 + i) for i, d in enumerate(synth.CLAHE_DISTS)])
    out = m.clahe_u8(dev(batch), 4, (8, 8)).cpu().numpy()
    for i in range(batch.shape[0]):
        assert np.array_equal(out[i], oracle.clahe_u8(batch[i], 4, 8, 8))
    chan = (synth.image_u8((200, 150), "gamma", 78).astype(np.float32) + np.float32(0.37)) / np.float32(255.3)
    assert np.array_equal(m.ChannelClahe(4, 8).apply(chan), g["channelclahe_200x150"])
    assert np.array_equal(m.ChannelClahe("4", "8").apply(chan), g["channelclahe_200x150"])      # string args from the mini-language
    cv2 = pytest.importorskip("cv2")
    for hw, grid, clip in (((3, 5), (8, 8), 4), ((50, 70), (5, 3), 4), ((64, 48), (8, 8), 0), ((2, 3), (8, 8), 4), ((2048, 33), (8, 8), 4)):
        im = synth.image_u8(hw, "bimodal", 600 + hw[0])
        ref = cv2.createCLAHE(clipLimit=clip, tileGridSize=grid).apply(im)
        assert np.array_equal(m.clahe_u8(dev(im), clip, grid).cpu().numpy(), ref), (hw, grid, clip)


def test_image_clahe_on_device(m, golden):
    cv2 = pytest.importorskip("cv2")
    g = golden("clahe")
    rgb = (np.random.RandomState(79).rand(90, 122, 3) ** 2.2).astype(np.float32)
    out = m.image_clahe(dev(rgb), 4, (8, 8)).cpu().numpy()
    np.testing.assert_allclose(out, g["imageclahe_90x122"], rtol=0, atol=2e-5)         # the reference's own output
    lat = oracle.cv2_lab_lattice()
    np.testing.assert_allclose(out, oracle.image_clahe(rgb, 4, 8, lat), rtol=0, atol=2e-5)
    # ragged batch, one launch per stage; sizes not divisible by 8
    rs = np.random.RandomState(80)
    imgs = [(rs.rand(h, w, 3) ** 3).astype(np.float32) for h, w in ((37, 53), (128, 96), (65, 200))]
    imgs[1][:8, :8] = 1.0
    imgs[1][8:16, :8] = 0.0
    outs = m.image_clahe([dev(i) for i in imgs], 4, (8, 8))
    for im, o in zip(imgs, outs):
        spc = (cv2.cvtColor(im, cv2.COLOR_RGB2LAB) + np.array([0, 128, 128], np.float32)) / np.array([100.0, 255.0, 255.0], np.float32)
        spc[:, :, 0] = oracle.channel_clahe(spc[:, :, 0], 4, 8)
        ref = cv2.cvtColor(spc * np.array([100.0, 255.0, 255.0], np.float32) - np.array([0, 128, 128], np.float32), cv2.COLOR_LAB2RGB)
        np.testing.assert_allclose(o.cpu().numpy(), ref, rtol=0, atol=2e-5)


def test_apply_clahe_transform(m):
    cv2 = pytest.importorskip("cv2")
    rs = np.random.RandomState(3)
    pic = (rs.rand(120, 160, 3) ** 3).astype(np.float32)
    out = m.ApplyClahe("4", "lab", "8")(pic)
    assert isinstance(out, list) and out[0].shape == pic.shape
    # reference arithmetic restated with cv2 for the colour conversion + the oracle CLAHE
    spc = (cv2.cvtColor(pic, cv2.COLOR_RGB2LAB) + np.array([0, 128, 128], np.float32)) / np.array([100.0, 255.0, 255.0], np.float32)
    spc[:, :, 0] = oracle.channel_clahe(spc[:, :, 0], 4, 8)
    ref = cv2.cvtColor(spc * np.array([100.0, 255.0, 255.0], np.float32) - np.array([0, 128, 128], np.float32), cv2.COLOR_LAB2RGB)
    np.testing.assert_allclose(out[0], ref, rtol=0, atol=2e-5)          # Lab<->RGB now runs on the device too
    two = m.CreateClahedImage()(pic)
    assert len(two) == 2 and np.allclose(two[1], ref, rtol=0, atol=2e-5)
    four = m.AddClaheFromRgb()(pic)[0]
    assert four.shape == (120, 160, 4)


def test_transform_classes_match_reference_registry(m, golden):
    """tests/golden/transforms.npz: outputs of the reference's TRANSFORMS['apply_clahe' | 'create_clahed' |
    'add_clahe_fromrgb'] built from the mini-language's string arguments; same calls on the drop-in classes."""
    g = golden("transforms")
    pic = g["pic"]
    np.testing.assert_allclose(m.ApplyClahe("4", "lab", "8")(pic.copy())[0], g["apply_clahe_4_lab_8"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(m.ApplyClahe("2", "lab", "4")(pic.copy())[0], g["apply_clahe_2_lab_4"], rtol=0, atol=2e-5)
    two = m.CreateClahedImage()(pic.copy())
    assert len(two) == 2 and np.array_equal(two[0], pic)
    np.testing.assert_allclose(two[1], g["create_clahed_1"], rtol=0, atol=2e-5)
    for args, key in (((), "add_clahe_fromrgb"), (("2", "4"), "add_clahe_fromrgb_2_4")):
        four = m.AddClaheFromRgb(*args)(pic.copy())
        assert isinstance(four, list) and len(four) == 1 and four[0].dtype == np.float32
        assert np.array_equal(four[0], g[key])                      # L channel: integer lattice + bit-exact CLAHE
    with pytest.raises(NotImplementedError):
        m.ApplyClahe("4", "luv", "8")(pic.copy())


# ------------------------------------------------------------------ ranks / top-k on the reference's scores
def test_ranks_from_reference_scores_bit_exact(m, golden):
    g = golden("search")
    assert np.array_equal(m.ranks_from_scores(g["scores"]).cpu().numpy(), g["ranks_stable"])
    assert np.array_equal(m.ranks_from_scores(g["scores_ties"]).cpu().numpy(), g["ranks_ties_stable"])
    for k in (1, 17, 100, 500):
        idx, val = m.topk_from_scores(g["scores_ties"], k)
        assert np.array_equal(idx.cpu().numpy(), g["ranks_ties_stable"][:k])
        assert np.array_equal(val.cpu().numpy(), np.take_along_axis(g["scores_ties"], g["ranks_ties_stable"][:k], 0))


def test_ranks_nan_rows_and_empty(m):
    # missing images give NaN descriptor rows in the reference (SURVEY.md section 5): np.argsort(-scores)
    # ranks them last in index order
    rs = np.random.RandomState(4)
    sc = rs.randn(3000, 5).astype(np.float32)
    sc[[7, 100, 2999], :] = np.nan
    sc[5, 2] = np.nan
    ref = oracle.ranks_from_scores(sc)
    assert np.array_equal(m.ranks_from_scores(sc).cpu().numpy(), ref)
    idx, val = m.topk_from_scores(sc, 10)
    assert np.array_equal(idx.cpu().numpy(), ref[:10])
    # NaN database rows never enter a top-k
    db = synth.descriptors(20000, 64, 5)
    db[[3, 77, 19999]] = np.nan
    q, src = synth.planted_queries(db[100:], 6, 9)
    index = m.Index(db, device=DEV)
    s, i = index.search(q, 50, precision="bf16")
    assert not np.isnan(s.cpu().numpy()).any() and np.array_equal(i.cpu().numpy()[:, 0], src + 100)
    # empty query batch
    s0, i0 = index.search(np.zeros((0, 64), np.float32), 10)
    assert tuple(s0.shape) == (0, 10) and tuple(i0.shape) == (0, 10)


def test_ranks_edge_cases(m):
    rs = np.random.RandomState(8)
    for n_db, n_q in ((1, 1), (2, 3), (4096, 2), (4097, 5), (12345, 33), (70000, 3)):
        sc = rs.randn(n_db, n_q).astype(np.float32)
        sc[rs.rand(n_db, n_q) < 0.3] = 0.5                        # heavy ties
        sc[0, 0] = -0.0
        if n_db > 1:
            sc[1, 0] = 0.0
        if n_db > 3:
            sc[2, 0] = np.inf
            sc[3, 0] = -np.inf
        ref = oracle.ranks_from_scores(sc)
        assert np.array_equal(m.ranks_from_scores(sc).cpu().numpy(), ref), (n_db, n_q)
        assert np.array_equal(m.ranks_from_scores(sc, method="radix").cpu().numpy(), ref), (n_db, n_q)


def test_ranks_constant_rows_with_infinities(m):
    """A constant score row has no finite spread: the histogram sort's scale is 0 and (hi - inf) * 0 would be NaN -- such
    queries must be handed to the sample sort whatever their length (found by the CPU property test of the plan)."""
    for n_db in (1500, 3000, 4096, 9000):
        sc = np.full((n_db, 4), 0.25, dtype=np.float32)
        sc[[3, 700, n_db - 1], 0] = np.inf
        sc[[5, 9], 1] = -np.inf
        sc[[1, 2, 1000], 2] = [np.inf, -np.inf, np.nan]
        sc[:, 3] = np.inf
        assert np.array_equal(m.ranks_from_scores(sc).cpu().numpy(), oracle.ranks_from_scores(sc)), n_db


@pytest.mark.parametrize("case", ["gauss", "gauss_outliers", "all_equal", "ascending", "descending", "periodic", "two_values", "spike", "heavy_tail"])
@pytest.mark.parametrize("n_db", [1024, 1025, 4993, 100000, 102400, 102401, 131072, 131073])
def test_ranks_sort_paths_distributions(m, case, n_db):
    """The three ranking routes against the stable argsort on distributions chosen to stress them.  Histogram sort
    (mdir_rank_scores_hist: 4096 cells linear in the score over mean +- 4 sigma of a strided sample): smooth populations,
    outliers far outside the range, +-inf / NaN / +-0, monotone data, heavy tails.  Sample sort (mdir_rank_scores_fast:
    splitters from a systematic sample, composite (score, row) keys): what the histogram sort flags -- massive ties,
    two-valued data, a dense spike -- plus data periodic in the row index (aliases with the systematic sample).
    Whatever the plans do, the result is exact: a bucket that cannot be staged falls through to the next route, the
    segmented radix sort last."""
    from mdir_b200 import search
    rs = np.random.RandomState(n_db % 1000 + len(case))
    n_q = 3
    i = np.arange(n_db, dtype=np.float64)
    if case == "gauss":
        sc = rs.randn(n_db, n_q) * 0.05
    elif case == "gauss_outliers":
        sc = rs.randn(n_db, n_q) * 0.03
        sc[rs.randint(0, n_db, 40), rs.randint(0, n_q, 40)] = rs.rand(40) * 2 - 1          # planted neighbours / far negatives
        sc[[0, 1, 2, 3, 4, 5], 0] = [np.inf, -np.inf, np.nan, 0.0, -0.0, np.nan]
    elif case == "all_equal":
        sc = np.full((n_db, n_q), 0.25)
    elif case == "ascending":
        sc = np.repeat((i / n_db)[:, None], n_q, 1)
    elif case == "descending":
        sc = np.repeat((-i / n_db)[:, None], n_q, 1)
    elif case == "periodic":
        period = max(2, n_db // (32 * max(1, -(-n_db // 400))))            # the sampling stride of the splitter kernel
        sc = np.stack([np.sin(2 * np.pi * i / period), (i % period) / period, ((i * 7) % period) / period], 1)
    elif case == "two_values":
        sc = (rs.rand(n_db, n_q) < 0.999).astype(np.float64)
    elif case == "heavy_tail":
        sc = rs.standard_cauchy((n_db, n_q)) * 0.01
    else:
        sc = rs.randn(n_db, n_q) * 1e-3
        sc[rs.rand(n_db, n_q) < 0.9] = 0.7
    sc = sc.astype(np.float32)
    before = dict(search.RANK_STATS)
    got = m.ranks_from_scores(sc).cpu().numpy()
    assert np.array_equal(got, oracle.ranks_from_scores(sc)), (case, n_db)
    if case in ("gauss", "gauss_outliers", "all_equal", "ascending", "descending", "two_values", "spike"):
        assert search.RANK_STATS["fallback"] == before["fallback"], "the radix fallback was needed on %s" % case
    if case in ("gauss", "gauss_outliers", "ascending", "descending") and 1025 <= n_db <= 131072:
        assert search.RANK_STATS["sample_sort"] == before["sample_sort"], "the histogram sort flagged %s" % case
    if case in ("all_equal", "two_values", "spike") and 4096 < n_db <= 131072:        # up to 4096 rows are one bucket, ties or not
        assert search.RANK_STATS["sample_sort"] == before["sample_sort"] + 1, "the histogram sort should hand %s to the sample sort" % case


# ------------------------------------------------------------------ similarity + search
def test_scores_and_drop_in_rank(m, golden):
    g = golden("search")
    db = synth.descriptors(500, 64, 11, clusters=20)
    q, _ = synth.planted_queries(db, 12, 12)
    index = m.Index(db, device=DEV)
    sc = index.scores(q).cpu().numpy()                            # (N_q, N_db)
    np.testing.assert_allclose(sc.T, g["scores"], rtol=0, atol=2e-3)
    # fp32 search == reference top-k wherever the reference's own gap exceeds fp32 noise
    s, i = index.search(q, 50, precision="fp32", shortlist=200)
    ref_i, ref_v = oracle.topk_from_scores(g["scores"], 66)       # 16 rows past k: the boundary swap rule needs them
    np.testing.assert_allclose(s.cpu().numpy().T, ref_v[:50], rtol=0, atol=2e-6)
    _assert_same_order(i.cpu().numpy().T, ref_i, ref_v, 2e-6)
    # the drop-in: (D,N) host matrices -> (N_db,N_q) int64 ranks -> the reference's compute_map
    ranks = m.rank(np.ascontiguousarray(db.T), np.ascontiguousarray(q.T))
    assert ranks.dtype == np.int64 and ranks.shape == (500, 12) and ranks.flags["C_CONTIGUOUS"]
    assert np.array_equal(np.sort(ranks, axis=0), np.tile(np.arange(500)[:, None], (1, 12)))     # each column a permutation
    gnd = synth.gnd_okjunk(500, 12, 13, empty_every=5)
    mp, aps, _, _ = oracle.compute_map(ranks, gnd, [1, 5, 10])
    assert abs(mp - float(g["okjunk_map"])) < 0.01
    avg, _, _ = oracle.compute_map_emh(ranks, synth.gnd_emh(500, 12, 14))
    for k_ in avg:
        assert abs(avg[k_] - float(g["emh_" + k_])) < 0.01


def test_tf32_and_fp32_faithful_scores(m, golden):
    g = golden("search")
    db = synth.descriptors(500, 64, 11, clusters=20)
    q, _ = synth.planted_queries(db, 12, 12)
    index = m.Index(db, device=DEV)
    np.testing.assert_allclose(index.scores(q, precision="tf32").cpu().numpy().T, g["scores"], rtol=0, atol=2e-3)
    s32 = index.scores(q, precision="fp32").cpu().numpy().T
    np.testing.assert_allclose(s32, g["scores"], rtol=0, atol=2e-6)                    # fp32-faithful (3xTF32)
    ranks = index.ranks(q, precision="fp32").cpu().numpy()
    _assert_same_order(ranks, g["ranks_stable"], np.take_along_axis(g["scores"], g["ranks_stable"], 0), 4e-6)
    # larger, non-multiple-of-32 dimension, several query blocks
    db2 = synth.descriptors(3000, 136, 31)
    q2 = synth.descriptors(150, 136, 32)
    idx2 = m.Index(db2, device=DEV)
    ref = oracle.scores(db2.T, q2.T)
    np.testing.assert_allclose(idx2.scores(q2, precision="fp32").cpu().numpy().T, ref, rtol=0, atol=2e-6)
    np.testing.assert_allclose(idx2.scores(q2, precision="tf32").cpu().numpy().T, ref, rtol=0, atol=2e-3)
    np.testing.assert_allclose(idx2.scores(q2, precision="bf16").cpu().numpy().T, ref, rtol=0, atol=2e-3)


@pytest.mark.parametrize("n_db,n_q,D", [(777, 129, 64), (5000, 300, 128), (33000, 1024, 64), (100, 257, 512)])
def test_dense_scores_one_launch_equals_per_block_launches(m, n_db, n_q, D):
    """mdir_sim_scan_dense_bf16 ((tile, 128-query block) work items, one launch) against one mdir_sim_scan_bf16 launch per
    128-query block: the same MMAs in the same order, so the scores are bit-identical; ragged last block and last tile."""
    import torch
    db = synth.descriptors(n_db, D, 3)
    q = synth.descriptors(n_q, D, 4)
    index = m.Index(db, device=DEV, keep_fp32=False)
    one = index.scores(q, precision="bf16")
    ref = torch.full((n_q, n_db), float("nan"), device=DEV)
    for q0 in range(0, n_q, 128):
        ref[q0:q0 + 128] = index.scores(q[q0:q0 + 128], precision="bf16")
    assert torch.equal(one, ref)
    assert np.abs(one.cpu().numpy() - (q @ db.T)).max() < 2e-3
    # a pitched output (column block of a wider array)
    wide = torch.zeros((n_q, n_db + 8), device=DEV)
    index.scores(q, out=wide[:, :n_db], precision="bf16")
    assert torch.equal(wide[:, :n_db], ref) and float(wide[:, n_db:].abs().max()) == 0.0


@pytest.mark.parametrize("n_db,n_q,D,k", [(70000, 300, 64, 10), (120000, 1024, 128, 10), (40000, 1500, 64, 100), (3000, 700, 64, 10)])
def test_wide_search_equals_per_block_search(m, n_db, n_q, D, k):
    """search(block_q=1024): SAMPLE and FILTER scans as ONE wide launch per 1,024 queries ((tile, 128-query block) work
    items, per-query filter state of all the blocks in shared memory) against the 128-queries-per-pass route: identical
    indices and scores, both precisions; ragged last block, several wide passes, the dense route of a small database."""
    import torch
    db = synth.descriptors(n_db, D, 5, clusters=40)
    q = synth.descriptors(n_q, D, 6)
    index = m.Index(db, device=DEV)
    index.fused = False                                    # the three-launch route for both (the one-launch route is <= 128 queries)
    for prec in ("bf16", "fp32"):
        s_ref, i_ref = index.search(q, k, precision=prec)
        s_w, i_w = index.search(q, k, precision=prec, block_q=1024)
        assert torch.equal(i_w, i_ref) and torch.equal(s_w, s_ref), prec
    ref_i, ref_v = oracle.topk_from_scores(oracle.scores(db.T, q[:64].T), k)
    assert (i_w[:64].cpu().numpy().T == ref_i).mean() > 0.99


def _assert_same_order(got, ref_i, ref_v, tol):
    """got (k, nq) vs the reference ranking ref_i / ref_v (k_ref >= k rows, best first): every position where the
    indices differ must hold a row that the REFERENCE places within `tol` of that position's reference score
    (summation-order noise between two fp32 dot products) -- including the last position, which is why callers pass a
    reference a few rows longer than k."""
    k, nq = got.shape
    assert ref_i.shape[0] >= k
    for j in range(nq):
        for r in range(k):
            if got[r, j] != ref_i[r, j]:
                near = np.abs(ref_v[:, j] - ref_v[r, j]) <= tol
                assert got[r, j] in ref_i[near, j], (r, j, got[r, j], ref_i[r, j])


@pytest.mark.parametrize("n_db,n_q,D,k", [(300, 5, 64, 10), (20000, 70, 256, 100), (16389, 128, 136, 64), (70000, 200, 64, 100), (50, 3, 8, 100)])
def test_search_bf16_equals_topk_of_own_scores(m, n_db, n_q, D, k):
    db = synth.descriptors(n_db, D, 100 + n_q, clusters=50)
    q, src = synth.planted_queries(db, n_q, 7)
    index = m.Index(db, device=DEV, idx_base=1000)
    sc = index.scores(q).cpu().numpy().T                          # (N_db, N_q) of the same bf16 path
    s, i = index.search(q, k, precision="bf16")
    ref_i, ref_v = oracle.topk_from_scores(sc, min(k, n_db))
    kk = min(k, n_db)
    assert np.array_equal(i.cpu().numpy().T[:kk], ref_i + 1000)
    assert np.array_equal(s.cpu().numpy().T[:kk], ref_v)
    if k > n_db:
        assert np.all(i.cpu().numpy()[:, n_db:] == -1) and np.all(np.isneginf(s.cpu().numpy()[:, n_db:]))
    assert np.all(i.cpu().numpy()[:, 0] == src + 1000)            # planted neighbour found first


@pytest.mark.parametrize("n_db,n_q,D,k", [(16389, 70, 64, 100), (120000, 128, 64, 132), (300000, 33, 32, 10)])
def test_search_one_launch_and_three_launch_routes_agree(m, n_db, n_q, D, k):
    """The fused threshold+filter launch and the sample -> select -> filter chain are both exact."""
    db = synth.descriptors(n_db, D, 300 + n_q, clusters=80)
    q, _ = synth.planted_queries(db, n_q, 9)
    index = m.Index(db, device=DEV, keep_fp32=False)
    assert index._fused_ok(k)
    sc = index.scores(q).cpu().numpy().T
    ref_i, ref_v = oracle.topk_from_scores(sc, k)
    for fused in (True, False, True):
        index.fused = fused
        s, i = index.search(q, k, precision="bf16")
        assert np.array_equal(i.cpu().numpy().T, ref_i), fused
        assert np.array_equal(s.cpu().numpy().T, ref_v), fused


def test_search_fp32_matches_reference_topk(m):
    db = synth.descriptors(30000, 128, 41, clusters=200)
    q, _ = synth.planted_queries(db, 70, 42)
    index = m.Index(db, device=DEV)
    s, i = index.search(q, 100, precision="fp32")
    sc = oracle.scores(db.T, q.T)
    ref_i, ref_v = oracle.topk_from_scores(sc, 116)
    np.testing.assert_allclose(s.cpu().numpy().T, ref_v[:100], rtol=0, atol=3e-6)
    _assert_same_order(i.cpu().numpy().T, ref_i, ref_v, 3e-6)
    assert index.cert["uncertified"] == 0 and not index.check_overflow()      # every query carries the shortlist certificate


def test_search_overflow_recovery(m):
    # adversarial order: scores increase with the row index, so every tile beats the sample
    # threshold and the candidate lists overflow; the re-threshold loop must still be exact
    n_db, D = 40000, 64
    rs = np.random.RandomState(5)
    base = rs.randn(D).astype(np.float32)
    base /= np.linalg.norm(base)
    noise = rs.randn(n_db, D).astype(np.float32) * 0.01
    db = (np.linspace(0.1, 1.0, n_db, dtype=np.float32)[:, None] * base[None, :] + noise).astype(np.float32)
    q = np.stack([base, -base, base + 0.1 * rs.randn(D).astype(np.float32)]).astype(np.float32)
    index = m.Index(db, device=DEV)
    sc = index.scores(q).cpu().numpy().T
    s, i = index.search(q, 100, precision="bf16")
    ref_i, ref_v = oracle.topk_from_scores(sc, 100)
    assert np.array_equal(i.cpu().numpy().T, ref_i) and np.array_equal(s.cpu().numpy().T, ref_v)
    # duplicates: identical rows tie on score and must come back in index order
    dup = np.repeat(synth.descriptors(50, 64, 3), 400, axis=0)
    index = m.Index(dup, device=DEV)
    s, i = index.search(dup[:2], 500, precision="bf16")
    ref_i, _ = oracle.topk_from_scores(index.scores(dup[:2]).cpu().numpy().T, 500)
    assert np.array_equal(i.cpu().numpy().T, ref_i)


def test_sharded_merge_equals_single(m):
    from mdir_b200 import _lib
    db = synth.descriptors(50000, 64, 61, clusters=100)
    q, _ = synth.planted_queries(db, 70, 62)
    k = 100
    single = m.Index(db, device=DEV)
    s1, i1 = single.search(q, k, precision="bf16")
    for world in (2, 4, 8):
        keys = []
        for r in range(world):
            lo, hi = m.ShardedIndex.shard_bounds(db.shape[0], world, r)
            shard = m.Index(db[lo:hi], device=DEV, idx_base=lo)
            keys.append(shard.search(q, k, precision="bf16", return_keys=True)[2])
        allk = torch.stack(keys).permute(1, 0, 2).contiguous().view(70, world * k)
        cnt = torch.full((70,), world * k, dtype=torch.int32, device=DEV)
        out_s = torch.empty((70, k), dtype=torch.float32, device=DEV)
        out_i = torch.empty((70, k), dtype=torch.int32, device=DEV)
        _lib.check(_lib.lib().mdir_topk_finalize(_lib.ptr(allk), world * k, _lib.ptr(cnt), 1, world * k, 0, 70, k, _lib.ptr(out_s),
                                                 _lib.ptr(out_i), None, None, None, _lib.stream()))
        assert torch.equal(out_i, i1) and torch.equal(out_s, s1), world


def test_r1m_full_size_properties(m):
    # BASELINE config 4 at full size: 70 q x 1,001,001 x 2048.  Size-independent checks:
    # planted neighbours come back first; the fused top-100 equals the top-100 selected from a
    # dense scan of the same index; fp32 re-scoring returns exactly-recomputed scores.
    n_db, D, n_q, k = 1001001, 2048, 70, 100
    g = torch.Generator(device=DEV).manual_seed(4)
    db = torch.empty((n_db, D), dtype=torch.float32, device=DEV)
    for r0 in range(0, n_db, 65536):
        blk = torch.randn((min(65536, n_db - r0), D), device=DEV, generator=g)
        db[r0:r0 + blk.shape[0]] = blk / blk.norm(dim=1, keepdim=True)
    src = torch.randint(0, n_db, (n_q,), device=DEV, generator=g)
    q = db[src] + 0.5 * torch.randn((n_q, D), device=DEV, generator=g) / D ** 0.5
    q = q / q.norm(dim=1, keepdim=True)
    index = m.Index.from_packed(m.search.pack_bf16(db), db32=db)
    s, i = index.search(q, k, precision="bf16")
    assert torch.equal(i[:, 0].long(), src)
    dense = index.scores(q)                                       # (70, 1001001)
    idx2, val2 = m.topk_from_scores(dense.t().contiguous(), k)
    assert torch.equal(idx2.t().int(), i) and torch.equal(val2.t(), s)
    s32, i32 = index.search(q, k, precision="fp32")
    exact = (db[i32.long().view(-1)].view(n_q, k, D) * q[:, None, :]).sum(-1)
    assert torch.allclose(s32, exact, rtol=0, atol=2e-6)
    assert torch.all(s32[:, :-1] >= s32[:, 1:]) and torch.equal(i32[:, 0].long(), src)
    assert (s32 - s).abs().max().item() < 2e-3                   # bf16 scores within the stated tolerance


def test_graphed_search_replays(m):
    from mdir_b200.search import GraphedSearch
    db = synth.descriptors(40000, 128, 71, clusters=100)
    index = m.Index(db, device=DEV)
    gs = GraphedSearch(index, n_q=70, k=100)
    for seed in (1, 2, 3):
        q, src = synth.planted_queries(db, 70, seed)
        s, i = gs(torch.from_numpy(q).pin_memory())
        torch.cuda.synchronize()
        assert not gs.check_overflow()
        s2, i2 = index.search(q, 100)
        assert torch.equal(i, i2) and torch.equal(s, s2)
        assert np.array_equal(i.cpu().numpy()[:, 0], src)
    # split graphs on one GPU: pack + scan | finalize + certified re-score, private candidate workspace, capped scan grid
    for scan_ctas in (0, 140, 64):
        gsp = GraphedSearch(index, n_q=70, k=100, overlap=True, split=True, scan_ctas=scan_ctas)
        assert gsp.split and gsp.overlap
        for seed in (4, 5):
            q, src = synth.planted_queries(db, 70, seed)
            s, i = gsp(torch.from_numpy(q).pin_memory())
            torch.cuda.synchronize()
            s2, i2 = index.search(q, 100)
            assert not gsp.check_overflow() and torch.equal(i, i2) and torch.equal(s, s2), scan_ctas


# ------------------------------------------------------------------ batched extract_vectors (section 8f, f2)
class ImageRetrievalNet(torch.nn.Module):
    """Shaped like cirtorch's ImageRetrievalNet: features / pool / norm / meta, no whitening."""

    def __init__(self, m, pooling="gem", p=2.9137):
        super().__init__()
        nn = torch.nn
        self.features = nn.Sequential(nn.Conv2d(3, 32, 3, stride=2, padding=1), nn.ReLU(), nn.Conv2d(32, 64, 3, stride=2, padding=1), nn.ReLU())
        self.lwhiten, self.whiten = None, None
        self.pool = {"gem": lambda: m.GeM(p=p), "mac": m.MAC, "spoc": m.SPoC}[pooling]()
        self.norm = m.L2N()
        self.meta = {"pooling": pooling, "regional": False, "whitening": False, "out_channels": 64, "outputdim": 64}

    def forward(self, x):                                     # imageretrievalnet.py:93-115 without whitening
        o = self.norm(self.pool(self.features(x))).squeeze(-1).squeeze(-1)
        return o.permute(1, 0)


class CirNetwork:
    """Shaped like mdir's CirNetwork (learning/network.py:72-89): .model + per-stage wrapper compositions."""

    def __init__(self, model, comp):
        self.model, self.wrappers, self.stage = model, {"eval": comp}, "eval"


def test_batched_extract_vectors(m, golden):
    torch.manual_seed(3)
    net = ImageRetrievalNet(m).to(DEV).eval()
    rs = np.random.RandomState(6)
    imgs = [torch.from_numpy(rs.rand(3, h, w).astype(np.float32)) for h, w in ((64, 48), (57, 91), (128, 96), (40, 40), (33, 77))]
    feats = lambda x: net.features(x.to(DEV).unsqueeze(0)).float().cpu().numpy()
    # ImageRetrievalNet semantics: single scale (extract_ss) and multi-scale with explicit msp (extract_ms)
    with torch.no_grad():
        v1 = m.extract_vectors(net, imgs, None, None, ms=[1], msp=1, group=2)
        assert tuple(v1.shape) == (64, 5) and v1.device.type == "cpu"
        for i, im in enumerate(imgs):
            close(v1[:, i], oracle.net_tail(feats(im), "gem", 2.9137)[:, 0], rtol=2e-5, atol=1e-7)
        ms = [1, 1 / np.sqrt(2), 1 / 2]
        v3 = m.extract_vectors(net, imgs, None, None, ms=ms, msp=2.9137, group=4)
        for i, im in enumerate(imgs):
            x = im.to(DEV).unsqueeze(0)
            outs = []
            for s in ms:
                xs = x if s == 1 else torch.nn.functional.interpolate(x, scale_factor=s, mode="bilinear", align_corners=False)
                outs.append(oracle.net_tail(net.features(xs).float().cpu().numpy(), "gem", 2.9137)[:, 0])
            close(v3[:, i], oracle.aggregate_tensor(outs, 3, 64, 2.9137), rtol=2e-5, atol=1e-7)
        # mdir CirNetwork semantics: wrappers carry the scales (msp rule) and the Lw whitening
        g = golden("head")
        lw = {"m": g["lw_m"][:64], "P": g["lw_P"][:64, :64]}
        comp = types.SimpleNamespace(wrappers=[m.CirtorchWhiten(lw, 32, DEV), m.CirMultiscaleAggregation(True, DEV)])
        cirnet = CirNetwork(net, comp)
        vw = m.extract_vectors(cirnet, imgs, None, None, group=3, return_device=True)
        assert tuple(vw.shape) == (5, 32) and vw.is_cuda
        for i, im in enumerate(imgs):
            x = im.to(DEV).unsqueeze(0)
            fm = [net.features(torch.nn.functional.interpolate(x, scale_factor=s, mode="bilinear", align_corners=False)).float().cpu().numpy() for s in ms]
            close(vw[i], oracle.gem_head(fm, 2.9137, 1e-6, lw["m"], lw["P"], 32), rtol=5e-5, atol=5e-7)


def test_extract_vectors_matches_reference_extract_vectors(m, golden):
    """tests/golden/extract.npz: outputs of the live cirtorch extract_vectors (single- and multi-scale) for a seeded
    network; the same weights and the same input tensors through the batched device path."""
    g = golden("extract")
    p = float(g["p"])
    net = ImageRetrievalNet(m, "gem", p)
    nn = torch.nn
    net.features = nn.Sequential(nn.Conv2d(3, 16, 3, stride=2, padding=1), nn.ReLU(), nn.Conv2d(16, 48, 3, stride=2, padding=1), nn.ReLU())
    net.features.load_state_dict({k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w_")})
    net.meta.update(out_channels=48, outputdim=48)
    net = net.to(DEV).eval()
    imgs = [torch.from_numpy(g["input_%d" % i]) for i in range(6)]
    ms = [float(s) for s in g["ms"]]
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False            # the reference ran its convolutions in fp32 on the CPU
    try:
        with torch.no_grad():
            v_ss = m.extract_vectors(net, imgs, None, None, ms=[1], msp=1, group=4)
            v_ms = m.extract_vectors(net, imgs, None, None, ms=ms, msp=p, group=3)
            v_m1 = m.extract_vectors(net, imgs, None, None, ms=ms, msp=1, group=6)
            # mdir's CirNetwork pattern: the eval wrappers carry the scales (msp rule) and the Lw whitening
            lw = {"m": g["lw_m"], "P": g["lw_P"]}
            comp = types.SimpleNamespace(wrappers=[m.CirtorchWhiten(lw, 32, DEV), m.CirMultiscaleAggregation(True, DEV)])
            cirnet = CirNetwork(net, comp)
            v_wr = m.extract_vectors(cirnet, imgs, None, None, group=4, return_device=True)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    assert tuple(v_wr.shape) == (6, 32)
    close(v_wr, g["compose_wh32"], rtol=2e-4, atol=5e-6)
    assert tuple(v_ss.shape) == (48, 6)
    close(v_ss, g["vecs_ss"], rtol=1e-4, atol=2e-6)
    close(v_ms, g["vecs_ms"], rtol=1e-4, atol=2e-6)
    close(v_m1, g["vecs_ms_msp1"], rtol=1e-4, atol=2e-6)


# ------------------------------------------------------------------ mAP on the device (section 8f, f3)
def test_compute_map_device(m, golden):
    g = golden("search")
    ru = g["ranks_ref_unstable"]
    gnd = synth.gnd_okjunk(500, 12, 13, empty_every=5)
    mp, aps, pr, prs = m.compute_map(ru, gnd, [1, 5, 10])
    close(mp, g["okjunk_map"], rtol=1e-12)
    np.testing.assert_array_equal(np.isnan(aps), np.isnan(g["okjunk_aps"]))
    close(np.nan_to_num(aps), np.nan_to_num(g["okjunk_aps"]), rtol=1e-12)
    close(pr, g["okjunk_pr"], rtol=1e-12)
    close(np.nan_to_num(prs), np.nan_to_num(g["okjunk_prs"]), rtol=1e-12)
    avg, per = m.compute_map_and_print("roxford5k", dev(ru), synth.gnd_emh(500, 12, 14))
    for k_ in avg:
        close(avg[k_], g["emh_" + k_], rtol=1e-12)
    for k_ in per:
        close(np.nan_to_num(per[k_]), np.nan_to_num(g["emh_" + k_]), rtol=1e-12)
    # the CirDatasetAp replacement path: descriptors -> ranks -> mAP, all on the device
    from mdir_b200.score import rank_and_evaluate
    db = synth.descriptors(500, 64, 11, clusters=20)
    q, _ = synth.planted_queries(db, 12, 12)
    import io, contextlib
    with contextlib.redirect_stdout(io.StringIO()):
        avg2, _ = rank_and_evaluate("synth", torch.from_numpy(np.ascontiguousarray(db.T)), torch.from_numpy(np.ascontiguousarray(q.T)), gnd)
    assert abs(avg2["map"] - float(g["okjunk_map"])) < 0.01
    # larger than one 1024-row chunk, many positives / junk, vs the oracle
    rs = np.random.RandomState(3)
    n_db, n_q = 30011, 9
    ranks = np.stack([rs.permutation(n_db) for _ in range(n_q)], axis=1)
    gnd2 = synth.gnd_okjunk(n_db, n_q, 5, n_ok=300, n_junk=500)
    gnd2[4]["ok"] = []                                     # no positives -> NaN, excluded
    ref = oracle.compute_map(ranks, gnd2, [1, 5, 10, 100])
    got = m.compute_map(ranks, gnd2, [1, 5, 10, 100])
    close(got[0], ref[0], rtol=1e-12)
    close(np.nan_to_num(got[1]), np.nan_to_num(ref[1]), rtol=1e-12)
    close(got[2], ref[2], rtol=1e-12)
    close(np.nan_to_num(got[3]), np.nan_to_num(ref[3]), rtol=1e-12)


# ------------------------------------------------------------------ alpha-QE / DBA (parity unpinned: vs the restated definitions)
def test_qe_and_dba(m):
    from mdir_b200 import qe
    db = synth.descriptors(5000, 64, 21, clusters=40)
    q, _ = synth.planted_queries(db, 9, 22)
    index = m.Index(db, device=DEV)
    q2 = qe.expand_queries(index, q, alpha=3.0, n_qe=10).cpu().numpy()
    close(q2, oracle.alpha_qe(db, q, 3.0, 10), rtol=1e-4, atol=2e-6)
    s, i = qe.search_qe(index, q, 20)
    ref_i, ref_v = oracle.topk_from_scores(db @ oracle.alpha_qe(db, q, 3.0, 10).T, 20)
    np.testing.assert_allclose(s.cpu().numpy().T, ref_v, rtol=0, atol=1e-5)
    small = synth.descriptors(600, 64, 23, clusters=10)
    aug = qe.dba(m.Index(small, device=DEV), alpha=3.0, k_dba=5)
    close(aug.db32, oracle.dba(small, 3.0, 5), rtol=1e-4, atol=2e-6)


@pytest.mark.parametrize("n_db,n_q,D,k", [(3000, 5, 64, 10), (70000, 70, 64, 100), (300000, 33, 32, 1200), (20000, 128, 136, 64)])
def test_c_abi_topk_composite_equals_index_search(m, n_db, n_q, D, k):
    """mdir_sim_topk_bf16 (one C call: plan + pack + scan + select + finalize) == Index.search, every route."""
    import torch
    from mdir_b200 import _lib
    db = synth.descriptors(n_db, D, 400 + n_q, clusters=60)
    q, _ = synth.planted_queries(db, n_q, 11)
    dev = torch.device(DEV)
    index = m.Index(db, device=dev, idx_base=77)
    lib = _lib.lib()
    d_q = torch.tensor(q, device=dev)
    ws = torch.empty((lib.mdir_sim_topk_workspace_bytes(D),), dtype=torch.uint8, device=dev)
    for prec, routes in (("bf16", (0, 1)), ("fp32", (0,))):
        if prec == "fp32" and k > 1024:
            continue
        ref_s, ref_i = index.search(q, k, precision=prec)
        for route in routes:
            if route == 1 and n_db > 131072:
                continue
            o_s = torch.empty((n_q, k), dtype=torch.float32, device=dev)
            o_i = torch.empty((n_q, k), dtype=torch.int32, device=dev)
            o_k = torch.empty((n_q, k), dtype=torch.int64, device=dev)
            ovf = torch.ones((n_q,), dtype=torch.int32, device=dev)
            with torch.cuda.device(dev):
                _lib.check(lib.mdir_sim_topk_bf16(_lib.ptr(index.db16), _lib.ptr(index.db32) if prec == "fp32" else None,
                                                  _lib.ptr(index.stats()) if prec == "fp32" else None, n_db, _lib.ptr(d_q),
                                                  n_q, D, k, 0, 77, route, _lib.ptr(o_s), _lib.ptr(o_i), _lib.ptr(o_k), _lib.ptr(ovf),
                                                  _lib.ptr(ws), _lib.stream()), "mdir_sim_topk_bf16")
            assert int(ovf.sum().item()) == 0                     # no overflow and (fp32) every query certified
            assert torch.equal(o_i, ref_i) and torch.equal(o_s, ref_s), (prec, route)
            assert torch.equal((o_k & 0xffffffff).to(torch.int32), ref_i)


def test_c_abi_gem_head_composite_equals_retrieval_head(m, golden):
    import ctypes
    import torch
    from mdir_b200 import _lib
    g = golden("head")
    C = 128
    lw = {"m": g["lw_m"], "P": g["lw_P"]}
    hws = [[(32, 24), (23, 17), (16, 12)], [(24, 32), (17, 23), (12, 16)], [(8, 8), (6, 6), (4, 4)]]
    flat = []
    for i, hw in enumerate(hws * 4):                      # 12 ragged images x 3 scales
        flat += [dev(synth.fmap((1, C, h, w), 950 + 7 * i + s, "relu")) for s, (h, w) in enumerate(hw)]
    lib = _lib.lib()
    for dims, whiten in ((64, True), (C, True), (C, False)):
        head = m.RetrievalHead("gem", p=2.9137, whitening=lw if whiten else None, dimensions=dims if whiten else None, nscales=3, device=DEV)
        ref = head(flat)
        pm = head.pack(flat)
        out = torch.empty((12, dims), dtype=torch.float32, device=ref.device)
        ws = torch.empty((lib.mdir_gem_head_workspace_bytes(12, 3, C, dims if whiten else 0),), dtype=torch.uint8, device=ref.device)
        with torch.cuda.device(ref.device):
            _lib.check(lib.mdir_gem_head(0, ctypes.c_void_p(pm.base), _lib.ptr(pm.off), _lib.ptr(pm.hw), 12, 3, C, 0, 2.9137, 1e-6, head.msp,
                                         _lib.ptr(head.m) if whiten else None, _lib.ptr(head.P) if whiten else None,
                                         _lib.ptr(head.Px3) if whiten else None, dims if whiten else 0, _lib.ptr(out), _lib.ptr(ws), _lib.stream()),
                       "mdir_gem_head")
        assert torch.equal(out, ref), (dims, whiten)


def test_rescore_f32_entry_point(m):
    """mdir_rescore_f32 directly: exact fp32 dot products of a shortlist, as keys; out-of-shard / negative ids pad."""
    import torch
    from mdir_b200 import _lib
    from mdir_b200.search import keys_to_host
    n_db, D, n_q, kk, base = 700, 136, 9, 17, 1000
    db = synth.descriptors(n_db, D, 301)
    q = synth.descriptors(n_q, D, 302)
    rs = np.random.RandomState(303)
    idx = (rs.randint(0, n_db, size=(n_q, kk)) + base).astype(np.int32)
    idx[0, 0], idx[1, 3], idx[2, 5] = -1, base + n_db, base - 1           # padding, past the shard, before the shard
    dev = torch.device(DEV)
    d_db, d_q, d_idx = torch.tensor(db, device=dev), torch.tensor(q, device=dev), torch.tensor(idx, device=dev)
    keys = torch.empty((n_q, kk), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().mdir_rescore_f32(_lib.ptr(d_db), n_db, base, _lib.ptr(d_q), n_q, D, _lib.ptr(d_idx), kk, _lib.ptr(keys), _lib.stream()))
    sc, gi = keys_to_host(keys.cpu().numpy().view(np.uint64))
    bad = (idx < base) | (idx >= base + n_db)
    assert np.all(gi[bad] == -1) and np.all(np.isneginf(sc[bad]))
    ref = np.einsum("qkd,qd->qk", db[np.clip(idx - base, 0, n_db - 1)].astype(np.float64), q.astype(np.float64))
    assert np.array_equal(gi[~bad], idx[~bad])
    np.testing.assert_allclose(sc[~bad], ref[~bad], rtol=0, atol=2e-6)


def test_search_pipeline_matches_blocking_search(m):
    """Double-buffered serving loop (async H2D / graph replay / D2H): same answers, in order, as index.search."""
    import torch
    db = synth.descriptors(80000, 64, 171, clusters=100)
    index = m.Index(db, device=DEV)
    pipe = m.SearchPipeline(index, n_q=40, k=50)
    batches = [torch.from_numpy(synth.planted_queries(db, 40, 200 + b)[0]).pin_memory() for b in range(7)]
    got = [(s.copy(), i.copy()) for s, i in pipe.map(batches)]
    assert len(got) == 7
    for b, (s, i) in enumerate(got):
        rs, ri = index.search(batches[b], 50)
        assert np.array_equal(i, ri.cpu().numpy()) and np.array_equal(s, rs.cpu().numpy()), b
    # tickets: out-of-order collection inside the window, misuse is an error
    t0, t1 = pipe.submit(batches[0]), pipe.submit(batches[1])
    with pytest.raises(m.MdirError):
        pipe.submit(batches[2])
    s1, i1 = pipe.result(t1)
    s0, i0 = pipe.result(t0)
    assert np.array_equal(i0, got[0][1]) and np.array_equal(i1, got[1][1])
    with pytest.raises(m.MdirError):
        pipe.result(t0)
    # a step whose candidate segments overflow is redone exactly (adversarial row order, as in the recovery test)
    n_db, D = 40000, 64
    rs_ = np.random.RandomState(5)
    base = rs_.randn(D).astype(np.float32)
    base /= np.linalg.norm(base)
    adv = (np.linspace(0.1, 1.0, n_db, dtype=np.float32)[:, None] * base[None, :] + rs_.randn(n_db, D).astype(np.float32) * 0.01).astype(np.float32)
    q = np.stack([base, -base, base + 0.1 * rs_.randn(D).astype(np.float32)]).astype(np.float32)
    idx2 = m.Index(adv, device=DEV)
    pipe2 = m.SearchPipeline(idx2, n_q=3, k=100, precision="bf16")
    outs = [(s.copy(), i.copy()) for s, i in pipe2.map([q, q, q])]
    ref_i, ref_v = oracle.topk_from_scores(idx2.scores(q).cpu().numpy().T, 100)
    for s, i in outs:
        assert np.array_equal(i.T, ref_i) and np.array_equal(s.T, ref_v)


# ---- f4: hard-negative mining, whitening learning ----------------------------------------------------

def test_mining_matches_reference_create_epoch_tuples(m, golden):
    g = golden("mining")
    for case in range(3):
        t = "c%d_" % case
        nnum = int(g[t + "nnum"])
        pos, dist = m.mine_hard_negatives(g[t + "qvecs"], g[t + "poolvecs"], g[t + "qclusters"], g[t + "poolclusters"], nnum, device=DEV)
        assert np.array_equal(g[t + "idxs2images"][pos.cpu().numpy()], g[t + "nidxs"])
        np.testing.assert_allclose(dist.cpu().numpy().reshape(-1), g[t + "ndist"], rtol=0, atol=2e-6)
    # the reference-variable form (traindataset.py:242-267 as one call)
    clusters = np.arange(400) % 40
    qidxs = [int(np.where(clusters == c)[0][0]) for c in g["c0_qclusters"]]
    nidxs, ndist = m.search_hard_negatives(g["c0_qvecs"], g["c0_poolvecs"], qidxs, g["c0_idxs2images"], clusters, 5, device=DEV)
    assert nidxs == g["c0_nidxs"].tolist() and len(ndist) == 300


def test_mining_larger_pool_and_exhaustion(m):
    D, n_pool, n_q, nnum = 64, 6000, 333, 7
    pool = synth.descriptors(n_pool, D, 81, clusters=150)
    q, src = synth.planted_queries(pool, n_q, 82)
    rs = np.random.RandomState(83)
    pc = rs.randint(0, 400, n_pool).astype(np.int32)
    qc = pc[src]
    pos, dist = m.mine_hard_negatives(q.T.copy(), pool.T.copy(), qc, pc, nnum, device=DEV)
    ref_pos, ref_dist = oracle.mine_negatives(q.T, pool.T, qc, pc, nnum)
    pos = pos.cpu().numpy()
    # fp32 summation-order noise may swap near-equal scores: wherever the picks differ, the reference's own scores of
    # the two pool images must lie within 4e-6 of each other (a measured bound, not a quota of free mismatches)
    sc_ref = np.dot(pool, q.T)
    qi, ji = np.nonzero(pos != ref_pos)
    assert np.all(np.abs(sc_ref[pos[qi, ji], qi] - sc_ref[ref_pos[qi, ji], qi]) <= 4e-6), "mining picks differ outside fp32 noise"
    assert len(qi) <= 0.01 * pos.size
    got_c = pc[pos]
    assert not np.any(got_c == qc[:, None]) and all(len(set(r)) == nnum for r in got_c)
    same = (pos == ref_pos)
    np.testing.assert_allclose(dist.cpu().numpy()[same], ref_dist[same], rtol=0, atol=3e-6)
    # only 3 clusters besides the query's: the 4th negative does not exist
    pc3 = (np.arange(n_pool) % 4).astype(np.int32)
    with pytest.raises(IndexError):
        m.mine_hard_negatives(q.T.copy(), pool.T.copy(), np.zeros(n_q, np.int32), pc3, 4, device=DEV)
    p3, _ = m.mine_hard_negatives(q.T.copy(), pool.T.copy(), np.zeros(n_q, np.int32), pc3, 3, device=DEV)
    assert np.all(np.sort(pc3[p3.cpu().numpy()], axis=1) == np.array([1, 2, 3]))


@pytest.mark.parametrize("M,N,K,kxn", [(128, 128, 64, False), (37, 211, 1000, False), (300, 70, 5000, True), (32, 32, 20000, False),
                                       (257, 129, 17, True), (1, 1, 1, False)])
def test_gemm_f64_matches_numpy(m, M, N, K, kxn):
    import torch
    rs = np.random.RandomState(M + N)
    A = rs.randn(M, K)
    B = rs.randn(K, N) if kxn else rs.randn(N, K)
    a_sub, b_sub = rs.randn(M), rs.randn(B.shape[0])
    ref = 0.37 * (A - a_sub[:, None]) @ ((B - b_sub[:, None]) if kxn else (B - b_sub[:, None]).T)
    dev = torch.device(DEV)
    got = m.gemm_f64(torch.tensor(A, device=dev), torch.tensor(B, device=dev), kxn, alpha=0.37,
                     a_sub=torch.tensor(a_sub, device=dev), b_sub=torch.tensor(b_sub, device=dev))
    np.testing.assert_allclose(got.cpu().numpy(), ref, rtol=0, atol=1e-12 * max(1.0, np.abs(ref).max()) * np.sqrt(K))
    got2 = m.gemm_f64(torch.tensor(A, device=dev), torch.tensor(B, device=dev), kxn)
    ref2 = A @ (B if kxn else B.T)
    np.testing.assert_allclose(got2.cpu().numpy(), ref2, rtol=0, atol=1e-12 * max(1.0, np.abs(ref2).max()) * np.sqrt(K))


def test_whitenlearn_matches_reference(m, golden):
    g = golden("whitenlearn")
    for case in range(2):
        t = "c%d_" % case
        N, D, seed, clusters = [int(x) for x in g[t + "X_recipe"]]
        X = synth.descriptors(N, D, seed, clusters=clusters).T.astype(np.float64)
        mm, P = m.whitenlearn(X, g[t + "qidxs"], g[t + "pidxs"], device=DEV)
        assert mm.shape == (D, 1) and P.shape == (D, D) and P.dtype == np.float64
        np.testing.assert_allclose(mm, g[t + "m"], rtol=0, atol=1e-13)
        scale = np.abs(g[t + "P"]).max()
        np.testing.assert_allclose(oracle.whitening_rows_aligned(P, g[t + "P"]), g[t + "P"], rtol=0, atol=1e-6 * scale)
        app = oracle.whitenapply(X[:, :50], mm, P)
        np.testing.assert_allclose(app.T @ app, g[t + "applied"].T @ g[t + "applied"], rtol=0, atol=1e-8)
        mp, Pp = m.pcawhitenlearn(X, device=DEV)
        np.testing.assert_allclose(mp, g[t + "pca_m"], rtol=0, atol=1e-13)
        np.testing.assert_allclose(oracle.whitening_rows_aligned(Pp, g[t + "pca_P"]), g[t + "pca_P"], rtol=0,
                                   atol=1e-6 * np.abs(g[t + "pca_P"]).max())
    # fp32 input (what extract_vectors hands over), shrinkage, and the learnt dict feeding the Lw head
    X32 = synth.descriptors(2000, 64, 91, clusters=40).T.copy()
    rs = np.random.RandomState(92)
    qi, pi = rs.randint(0, 2000, 500), rs.randint(0, 2000, 500)
    mm, P = m.whitenlearn(X32, qi, pi, device=DEV)
    mo, Po = oracle.whitenlearn(X32, qi, pi)
    np.testing.assert_allclose(mm, mo, rtol=0, atol=1e-12)
    np.testing.assert_allclose(oracle.whitening_rows_aligned(P, Po), Po, rtol=0, atol=1e-6 * np.abs(Po).max())
    mp, Pp = m.pcawhitenlearn(X32, shrink=10, device=DEV)
    mo, Po = oracle.pcawhitenlearn(X32, shrink=10)
    np.testing.assert_allclose(oracle.whitening_rows_aligned(Pp, Po), Po, rtol=0, atol=1e-6 * np.abs(Po).max())
    out = m.whitenapply(X32[:, :20].astype(np.float64), mm, P, 32)
    np.testing.assert_allclose(np.abs(out), np.abs(oracle.whitenapply(X32[:, :20].astype(np.float64), mm, P, 32)), rtol=0, atol=1e-5)


def test_bench_line_contract(tmp_path):
    """python bench.py (short run): one JSON line on stdout with the metric, roofline, cpu_baseline, e2e, clocks and
    gpu_launches objects the measurement contract asks for; --dump-outputs writes the last timed step's top-100."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dump = str(tmp_path / "dump")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "20", "--warmup", "3", "--no-extras", "--cpu-rows", "4000",
                          "--dump-outputs", dump], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-800:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["unit"] == "queries/s" and d["n_gpus"] == 1 and d["steps"] == 20 and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["dtype"] == "bf16" and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["value"] > 1e4 and abs(d["value"] - 70 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and 0.3 < r["frac"] < 1.3 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] > 0.9 * r["algorithmic_bytes_per_launch"]
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and c["unit"] == "queries/s" and c["sample"]
    e = d["e2e"]
    assert e["value"] > 1e4 and e["h2d_bytes_per_step"] == 70 * 2048 * 4 and e["d2h_bytes_per_step"] == 70 * 100 * 8 + 70 * 4
    pc = d["parity_check"]                                     # the timed graphs' results against the independent ranking
    assert pc["checked_queries"] == 8 * 70 and pc["mismatches"] == 0 and pc["certificate_failures"] == 0
    assert d["gpu_launches"] == 20 * 3                         # pack, fused scan, finalize+re-score per step
    assert "sm_mhz" in d["clocks"] or "error" in d["clocks"]
    sc, ix = np.load(os.path.join(dump, "scores.npy")), np.load(os.path.join(dump, "indices.npy"))
    assert sorted(os.listdir(dump)) == ["indices.npy", "scores.npy"]
    assert sc.shape == ix.shape == (70, 100) and sc.dtype == np.float32 and ix.dtype == np.float64
    assert np.all(np.isfinite(sc)) and np.all(np.diff(sc, axis=1) <= 0)            # best first
    assert np.all(ix == np.round(ix)) and ix.min() >= 0 and ix.max() < 1001001
    assert all(len(np.unique(row)) == 100 for row in ix)
    # the dump is the LAST timed step: query batch (20 - 1) % N_BATCHES of the seeded inputs, ranked independently here
    # (dense fp32 scores -> 148 candidates -> fp64 re-scoring), swaps accepted only inside 2e-6 gaps as in the bench
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    db32, q_host = bench.synthetic_inputs(torch, torch.device("cuda", 0), 0, bench.N_DB, 0)
    q = q_host[(20 - 1) % bench.N_BATCHES].to(db32.device)
    cand = torch.topk(q @ db32.T, 148, dim=1).indices
    v64 = (db32[cand].double() * q.double()[:, None, :]).sum(-1)
    r_i, r_v = cand.cpu().numpy(), v64.cpu().numpy()
    del db32, cand, v64
    order = np.lexsort((r_i, -r_v), axis=1)[:, :116]
    r_i, r_v = np.take_along_axis(r_i, order, 1), np.take_along_axis(r_v, order, 1)
    bad, _ = bench.same_topk(ix.astype(np.int64), sc.astype(np.float64), r_i, r_v, 2e-6)
    assert bad == 0
