"""CPU-side checks: the C-ABI library builds, loads and exports every symbol that
include/mdir_b200.h declares; host-side key/merge/shard logic; loud failure without CUDA;
registry patching by install() (only where the reference checkout is present)."""
import os
import re
import ctypes

import numpy as np
import pytest
import torch

from oracle import oracle, synth, ref_import

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def libpath():
    from mdir_b200 import build
    return build.build()


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "mdir_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mdir_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(libpath):
    names = declared_symbols()
    assert len(names) >= 18
    l = ctypes.CDLL(libpath)
    for n in names:
        assert hasattr(l, n), "missing export " + n
    from mdir_b200 import _lib
    assert sorted(_lib.PROTOTYPES) == names, "ctypes prototypes out of sync with the header"
    assert _lib.lib().mdir_abi_version() == _lib.ABI_VERSION


def test_key_helpers_match_c(libpath):
    from mdir_b200 import _lib
    from mdir_b200.search import make_keys_host, keys_to_host
    l = _lib.lib()
    rs = np.random.RandomState(0)
    s = np.concatenate([rs.randn(200).astype(np.float32), np.array([0.0, -0.0, 1e-40, -1e-40, np.inf, -np.inf], np.float32)])
    i = rs.randint(0, 2 ** 32 - 1, size=s.shape[0], dtype=np.int64)
    k = make_keys_host(s, i)
    for a, b, kk in zip(s, i, k):
        assert l.mdir_make_key(float(a), int(b)) == int(kk)
    sc, idx = keys_to_host(k)
    assert np.array_equal(sc, np.where(s == 0, np.float32(0), s)) and np.array_equal(idx, i)
    # key order == (score desc, index asc) == stable argsort of -scores
    sc2 = np.round(rs.randn(500) * 3).astype(np.float32) / 3
    keys = make_keys_host(sc2, np.arange(500))
    assert np.array_equal(np.argsort(keys, kind="stable"), oracle.ranks_from_scores(sc2[:, None])[:, 0])


def test_merge_keys_host_equals_global_topk():
    from mdir_b200.search import make_keys_host, keys_to_host, merge_keys_host, ShardedIndex
    db = synth.descriptors(1000, 32, 5, clusters=10)
    q, _ = synth.planted_queries(db, 9, 6)
    sc = oracle.scores(db.T, q.T)                      # (N, Nq)
    sc = np.round(sc * 50).astype(np.float32) / 50      # ties across shards
    k = 20
    for world in (1, 2, 4, 8):
        parts = []
        for r in range(world):
            lo, hi = ShardedIndex.shard_bounds(1000, world, r)
            idx, val = oracle.topk_from_scores(sc[lo:hi], min(k, hi - lo))
            keys = make_keys_host(val.T, idx.T + lo)
            pad = np.full((9, k), np.uint64(0xffffffffffffffff))
            pad[:, :keys.shape[1]] = keys
            parts.append(pad)
        merged = merge_keys_host(np.stack(parts), k)
        msc, midx = keys_to_host(merged)
        gidx, gval = oracle.topk_from_scores(sc, k)
        assert np.array_equal(midx, gidx.T) and np.array_equal(msc, gval.T), world


def test_shard_bounds_cover():
    from mdir_b200.search import ShardedIndex
    for n in (0, 1, 7, 1001001):
        for w in (1, 2, 4, 8):
            b = [ShardedIndex.shard_bounds(n, w, r) for r in range(w)]
            assert b[0][0] == 0 and b[-1][1] == n
            assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))


def test_module_surface_matches_reference_names():
    import mdir_b200
    g = mdir_b200.GeM(p=2.9137)
    assert repr(g) == "GeM(p=2.9137, eps=1e-06)"
    assert list(g.state_dict().keys()) == ["p"] and g.p.shape == (1,)
    assert repr(mdir_b200.MAC()) == "MAC()" and repr(mdir_b200.SPoC()) == "SPoC()"
    assert repr(mdir_b200.L2N()) == "L2N(eps=1e-06)"
    assert set(mdir_b200.POOLING) == {"gem", "mac", "spoc"}
    ms = mdir_b200.CirMultiscaleAggregation("True", "cpu")
    assert np.allclose(ms.scales, [1, 1 / np.sqrt(2), 0.5])
    assert mdir_b200.CirMultiscaleAggregation(False, "cpu").scales == [1]
    t, was = ms.preprocess(torch.zeros(1, 3, 64, 48), None)
    assert [tuple(x.shape[-2:]) for x in t] == [(64, 48), (45, 33), (32, 24)] and was is False


def test_no_cpu_fallback():
    import mdir_b200
    with pytest.raises(mdir_b200.MdirError):
        mdir_b200.gem(torch.zeros(1, 4, 3, 3))
    with pytest.raises(mdir_b200.MdirError):
        mdir_b200.l2n(torch.zeros(1, 4, 1, 1))
    with pytest.raises(mdir_b200.MdirError):
        mdir_b200.clahe_u8(torch.zeros(8, 8, dtype=torch.uint8))
    with pytest.raises(mdir_b200.MdirError):
        mdir_b200.Index(np.zeros((4, 8), np.float32), device="cpu")


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "mdir_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f


@pytest.mark.skipif(not ref_import.available(), reason="needs the mdir reference checkout (MDIR_REF_ROOT, oracle/_ref or baseline/_ref)")
def test_install_patches_registries():
    ref_import.import_reference()
    import mdir_b200
    patched = mdir_b200.install()
    import cirtorch.networks.imageretrievalnet as irn
    import mdir.components.data.wrapper as mwrap
    import mdir.components.data.transform as mtrans
    import mdir.components.optim.score as mscore
    assert irn.POOLING["gem"] is mdir_b200.GeM and irn.POOLING["mac"] is mdir_b200.MAC
    assert "rmac" in irn.POOLING                                   # untouched (out of scope)
    assert mwrap.WRAPPERS_LABELS["cirwhiten"] is mdir_b200.CirtorchWhiten
    assert mwrap.WRAPPERS_LABELS["cirmultiscale"] is mdir_b200.CirMultiscaleAggregation
    assert mtrans.TRANSFORMS["apply_clahe"].device_class is mdir_b200.ApplyClahe
    # colourspaces the device path does not cover stay the reference's own classes (functional.py:24-48)
    from mdir.components.data.transform import photometric_transforms as ref_pt
    assert isinstance(mtrans.TRANSFORMS["apply_clahe"]("4", "luv", "8"), ref_pt.ApplyClahe)
    assert isinstance(mtrans.TRANSFORMS["add_clahe_fromrgb"]("4", "8", "lsh"), ref_pt.AddClaheFromRgb)
    assert isinstance(mtrans.TRANSFORMS["apply_clahe"]("4", "lab", "8"), mdir_b200.ApplyClahe)
    mdir_b200.install()                                            # idempotent: the reference class is not lost
    assert mtrans.TRANSFORMS["apply_clahe"].reference_class is ref_pt.ApplyClahe
    assert mscore.SCORES["cirdatasetap"].__name__ == "CirDatasetAp"
    assert len(patched) >= 9
    # the yaml-driven wrapper factory builds ours (wrapper.py:209-220)
    comp = mwrap.initialize_wrappers({"1_cirmultiscale": {"scales": True}}, torch.device("cpu"))
    assert isinstance(comp.wrappers[0], mdir_b200.CirMultiscaleAggregation)


def _balanced_grid(n_work, max_ctas):
    """common.cuh:balanced_grid -- the smallest persistent grid that needs as many rounds as max_ctas CTAs would."""
    if n_work <= 0 or max_ctas <= 0:
        return 1
    if n_work <= max_ctas:
        return int(n_work)
    rounds = -(-n_work // max_ctas)
    return int(-(-n_work // rounds))


def _topk_plan_restatement(n_db, kth, sms):
    """The top-k route rules in Python, the reference mdir_topk_plan is checked against -> (route, n_sample, stride).
    Three-launch sampling plan: the threshold is the kth best of n_sample * 256 sampled rows, so about
    kth * n_tiles / n_sample rows survive the filter pass; n_sample is sized to keep that near 4,500 (None: no plan,
    dense).  One-launch route: each of the g persistent CTAs samples one tile, so the threshold is about the kth best
    of g * 256 rows and ~1.25 * kth * n_tiles / g rows survive, spread over g segments; taken when that keeps the
    segments at most half full.  Route 1 reports the three-launch plan too (the fallback of more than 128 queries)."""
    from mdir_b200 import search
    n_tiles = (n_db + search.TILE - 1) // search.TILE
    if n_tiles < 64:
        return 0, 0, 0
    want = -(-kth * n_tiles // 4500)                            # ceil
    if want > 148:                                              # whole waves of the 148 persistent CTAs
        want = -(-want // 148) * 148
    n_sample = max(32, min(search.MAX_SAMPLE_TILES, n_tiles // 4, want))
    stride = n_tiles // n_sample
    plan = (0, 0, 0) if n_sample * search.TILE < 2 * kth or stride < 2 else (2, n_sample, stride)
    g = _balanced_grid(n_tiles, min(148, sms, n_tiles // 2))
    if g * 16 >= 2 * kth and 1.25 * kth * n_tiles / (g * g) <= search.FUSED_CAP_L / 2:
        return (1,) + plan[1:]
    return plan


def test_topk_route_planner_c_equals_python(libpath):
    """mdir_topk_plan (composite.cu), the one planner of Index.search and mdir_sim_topk_bf16, equals the Python
    statement of the route rules for every database size / depth / SM count, sampling plan included; Index._route
    demotes the one-launch route to that plan when the route is disabled or a block has more than 128 queries."""
    import ctypes as C
    from mdir_b200 import search
    l = C.CDLL(libpath)
    l.mdir_topk_plan.argtypes = [C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    rs = np.random.RandomState(0)
    sizes = [1, 255, 16383, 16384, 16385, 20000, 32768, 75000, 125126, 250251, 1001001, 2600000, 4000000, 20000000]
    sizes += [int(x) for x in rs.randint(1, 5_000_000, 60)]
    routes = set()
    for n_db in sizes:
        for kth in (1, 10, 100, 132, 200, 384, 700, 1184, 1185, 2048, 4096):
            for sms in (148, 132, 60):
                want = _topk_plan_restatement(n_db, kth, sms)
                r, ns, st = C.c_int(-1), C.c_int(-1), C.c_int(-1)
                assert l.mdir_topk_plan(n_db, kth, sms, C.byref(r), C.byref(ns), C.byref(st)) == 0
                assert (r.value, ns.value, st.value) == want, (n_db, kth, sms, want, (r.value, ns.value, st.value))
                routes.add(want[0])
                idx = search.Index.__new__(search.Index)
                idx.n, idx._sms, idx.fused = n_db, sms, True
                assert idx._route(kth, 128) == want and idx._fused_ok(kth) == (want[0] == 1)
                demoted = want if want[0] != 1 else ((2,) + want[1:] if want[1] else (0, 0, 0))
                assert idx._route(kth, 129) == demoted
                idx.fused = False
                assert idx._route(kth, 1) == demoted and not idx._fused_ok(kth)
    assert routes == {0, 1, 2}


def test_tune_knobs_and_workspace_sizes_are_host_only(libpath):
    """Host-only entry points of the round-2 additions answer without a GPU: the SM-partition knobs validate their
    arguments, and the three ranking routes report workspace sizes that grow with the problem (the histogram sort
    needs a compact 8 B/pair array, the sample sort over-provisioned bucket regions)."""
    import ctypes as C
    l = C.CDLL(libpath)
    l.mdir_tune.argtypes = [C.c_int, C.c_int]
    assert l.mdir_tune(1, 98) == 0 and l.mdir_tune(1, 0) == 0
    assert l.mdir_tune(2, 0) == 0 and l.mdir_tune(2, 1) == 0
    assert l.mdir_tune(3, 4096) == 0 and l.mdir_tune(3, 0) == 0
    assert l.mdir_tune(2, 7) != 0 and l.mdir_tune(99, 0) != 0 and l.mdir_tune(1, -1) != 0
    for fn in ("mdir_rank_workspace_bytes", "mdir_rank_fast_workspace_bytes", "mdir_rank_hist_workspace_bytes"):
        f = getattr(l, fn)
        f.argtypes, f.restype = [C.c_int64, C.c_int], C.c_size_t
        assert f(0, 5) == 0 and f(100000, 0) == 0
        assert 0 < f(100000, 64) < f(100000, 128) < f(200000, 128)
    hist, fast = l.mdir_rank_hist_workspace_bytes, l.mdir_rank_fast_workspace_bytes
    assert hist(100000, 1024) >= 100000 * 1024 * 16                       # pairs 8 B + ranks 4 B + transposed scores 4 B
    assert hist(500, 8) == fast(500, 8) and hist(200000, 8) == fast(200000, 8)      # lengths the histogram sort forwards


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` runs on the host alone and prints exactly one JSON line with the contract's keys."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-rows", "3000"],
                         capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"]


def test_batched_extraction_is_whitelisted():
    """ADVICE r1 (high): the batched extractor must refuse every network it does not positively recognise -- a branched
    model (forward overridden, cirnet.py:25-45) or an unknown composite -- so that install()'s extractor falls back to the
    reference's per-image loop instead of silently evaluating `.model.features` alone; mdir's SequentialNetwork
    (normaliser -> CirNet, learning/network.py:204-236) IS understood: its earlier stages run on every scaled image."""
    from mdir_b200 import extract, score

    class ImageRetrievalNet(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.features = torch.nn.Identity()
            self.pool = type("GeM", (torch.nn.Module,), {})()
            self.pool.p = torch.nn.Parameter(torch.ones(1) * 3)
            self.pool.eps = 1e-6
            self.lwhiten = self.whiten = None
            self.meta = {"pooling": "gem", "regional": False, "whitening": False, "outputdim": 8, "out_channels": 8}

        def forward(self, x):
            return x

    class ImageRetrievalNetBranched(ImageRetrievalNet):
        def forward(self, x):
            return x + 1

    class Comp:
        wrappers = []

    class CirNetwork:
        def __init__(self, model):
            self.model, self.wrappers = model, {"eval": Comp()}

    class SingleNetwork(CirNetwork):
        pass

    class SequentialNetwork:
        def __init__(self, first, last):
            self.networks, self.sequence = {"a": first, "b": last}, ["a", "b"]
            self.model, self.wrappers = last.model, last.wrappers

    class SomethingElse(SequentialNetwork):
        pass

    base = ImageRetrievalNet()
    assert extract._Plan(base, [1], 1).pre == []
    assert extract._Plan(CirNetwork(base), [1], 1).model is base
    first = SingleNetwork(ImageRetrievalNet())
    plan = extract._Plan(SequentialNetwork(first, CirNetwork(base)), [1], 1)
    assert plan.pre == [first] and plan.model is base
    for bad in (ImageRetrievalNetBranched(), CirNetwork(ImageRetrievalNetBranched()), SomethingElse(first, CirNetwork(base)),
                SequentialNetwork(first, CirNetwork(ImageRetrievalNetBranched()))):
        with pytest.raises(NotImplementedError):
            extract._Plan(bad, [1], 1)
    # the installed extractor: unrecognised -> the reference loop (with DataLoader workers forced to 0), recognised -> ours
    calls = []
    ev = score._batched_or_reference(lambda *a, **k: calls.append(torch.utils.data.DataLoader([0], num_workers=6).num_workers) or "ref", True)
    assert ev(CirNetwork(ImageRetrievalNetBranched()), [], 10, None) == "ref" and calls == [0]
    assert torch.utils.data.DataLoader([0], num_workers=2).num_workers == 2            # restored afterwards
