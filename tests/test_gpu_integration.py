"""End-to-end integration (SURVEY.md App. B, section 4 "integration" row; VERDICT r1 rows g2 / a12): the reference's own
``mdir.stages.validate.validate(scenario, ())`` un-patched versus after ``mdir_b200.install()``, on the GPU box, with
the UNMODIFIED reference staged under baseline/_ref (baseline/stage_ref.py).  Each arm runs in its own process
(tools/integration_validate.py).  Bars: mAP reported by validate() equal to 0.01 against the reference on the CPU,
per-query AP equal to 0.01, descriptors equal to 1e-5 against the reference running the same backbone on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle, ref_import

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "tools", "integration_validate.py")
KINDS = ("c1", "c2", "c2seq")


def _run(*args, env=None):
    e = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    e.update(env or {})
    r = subprocess.run([sys.executable, TOOL] + list(args), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=e, timeout=900)
    assert r.returncode == 0, r.stdout.decode()[-4000:]
    return r.stdout.decode()


@pytest.fixture(scope="module")
def arms(tmp_path_factory):
    if not ref_import.available():
        pytest.skip("needs the mdir reference checkout (MDIR_REF_ROOT, oracle/_ref or baseline/_ref)")
    root = str(tmp_path_factory.mktemp("integ"))
    _run("fixture", root)
    out = {}
    for arm in ("ref_cpu", "ref_cuda", "ours", "ours_modules"):
        path = os.path.join(root, arm + ".npz")
        _run("run", root, arm, path)
        out[arm] = np.load(path, allow_pickle=False)
    out["root"] = root
    return out


def _gnd(root):
    db = open(os.path.join(root, "db.tsv")).read().split("\n")[1:-1]
    pos = {n: i for i, n in enumerate(db)}
    gnd = []
    for line in open(os.path.join(root, "q.tsv")).read().split("\n")[1:-1]:
        _, _, ok, junk = line.split("\t")
        gnd.append({"ok": [pos[x] for x in json.loads(ok)], "junk": [pos[x] for x in json.loads(junk)]})
    return gnd


def test_registries_select_our_modules(arms):
    """a12: the yaml `pooling: gem` key builds OUR GeM through init_cirnet / init_network (cirnet.py:10-22,
    imageretrievalnet.py:203), the wrapper mini-language builds OUR wrappers, and both run on the GPU."""
    for arm in ("ours", "ours_modules"):
        info = json.loads(str(arms[arm]["info"]))
        for kind in KINDS:
            assert info["%s_pool_module" % kind] == "mdir_b200.layers.GeM", info
            assert info["%s_device" % kind].startswith("cuda")
        assert info["c2_wrappers"] == ["mdir_b200.wrappers.CirtorchWhiten", "mdir_b200.wrappers.CirMultiscaleAggregation"]
        assert "SCORES[cirdatasetap]" in info["patched"] and "POOLING[gem]" in info["patched"]
    info = json.loads(str(arms["ref_cuda"]["info"]))
    assert info["c1_pool_module"] == "cirtorch.layers.pooling.GeM" and info["c1_device"].startswith("cuda")
    assert json.loads(str(arms["ref_cpu"]["info"]))["cuda"] is False


@pytest.mark.parametrize("kind", KINDS)
def test_validate_map_matches_reference(arms, kind):
    gnd = _gnd(arms["root"])
    ref = arms["ref_cpu"]
    ref_map = float(ref[kind + "_map"][0])
    ref_aps = oracle.compute_map(oracle.ranks(ref[kind + "_vecs"], ref[kind + "_qvecs"]), gnd)[1]
    assert abs(ref_map - np.nanmean(ref_aps)) < 1e-9               # the oracle restates what validate() reported
    for arm in ("ref_cuda", "ours", "ours_modules"):
        got = arms[arm]
        assert abs(float(got[kind + "_map"][0]) - ref_map) <= 0.01, (arm, kind, float(got[kind + "_map"][0]), ref_map)
        aps = oracle.compute_map(oracle.ranks(got[kind + "_vecs"], got[kind + "_qvecs"]), gnd)[1]
        np.testing.assert_allclose(aps, ref_aps, rtol=0, atol=0.01, err_msg="%s %s per-query AP" % (arm, kind))


@pytest.mark.parametrize("kind", KINDS)
def test_descriptors_match_reference(arms, kind):
    """Same backbone arithmetic (the reference on cuda:0): what differs is only our head (and, in c2 / c2seq, our CLAHE
    transform in the `ours` arm, whose RGB output is within 2e-5 of OpenCV's).  Unit-norm descriptors, absolute tolerance."""
    ref = arms["ref_cuda"]
    for arm in ("ours", "ours_modules"):
        for key in ("_vecs", "_qvecs"):
            a, b = arms[arm][kind + key], ref[kind + key]
            assert a.shape == b.shape and a.dtype == np.float32
            tol = 1e-5 if (arm == "ours_modules" or kind == "c1") else 2e-4       # GPU CLAHE pixels differ by <= 2e-5 upstream of the CNN
            assert np.abs(a - b).max() <= tol, (arm, kind, key, float(np.abs(a - b).max()))
    # and against the CPU oracle the whole pipeline (CPU vs GPU convolutions included) stays close
    for key in ("_vecs", "_qvecs"):
        assert np.abs(arms["ours"][kind + key] - arms["ref_cpu"][kind + key]).max() <= 1e-3
