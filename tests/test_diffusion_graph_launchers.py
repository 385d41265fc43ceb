"""CPU-side checks of captured diffusion serving: mdir_diffusion_solve_dev / mdir_diffusion_combine_dev refuse NULL
required pointers and out-of-range parameters before touching the device, their ctypes prototypes match the header,
and GraphedDiffusion / DiffusionPipeline validate their source and parameters without a GPU."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = C.c_void_p(256)          # a non-NULL pointer the launchers must never dereference on the host
NULL = C.c_void_p(0)
CTYPES = {"int": C.c_int, "int64_t": C.c_int64, "float": C.c_float, "double": C.c_double, "size_t": C.c_size_t}


@pytest.fixture(scope="module")
def lib():
    from mdir_b200 import build, _lib
    build.build()
    return _lib.lib()


def header_argtypes(name):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "mdir_b200.h")).read(), flags=re.S)
    m = re.search(r"\bint\s+%s\s*\(([^)]*)\)" % name, text)
    assert m, name
    out = []
    for arg in m.group(1).split(","):
        arg = " ".join(arg.split())
        out.append(C.c_void_p if "*" in arg else CTYPES[arg.rsplit(" ", 1)[0]])
    return out


@pytest.mark.parametrize("name", ["mdir_diffusion_solve_dev", "mdir_diffusion_combine_dev"])
def test_prototypes_match_header(name):
    from mdir_b200 import _lib
    res, args = _lib.PROTOTYPES[name]
    assert res is C.c_int and args == header_argtypes(name)


def solve_dev(lib, **kw):
    a = dict(L_ids=P, L_s=P, n_q=4, trunc=1000, slot_id=P, n_used=20000, nbr=P, S=P, k=50, k_q=10, gamma=3.0, alpha=0.99,
             iters=20, rtol=1e-6, k_out=100, ws=P, ws_bytes=0, f_out=P, ids_out=P, n_used_dev=P, status=P, stream=NULL)
    a.update(kw)
    return lib.mdir_diffusion_solve_dev(*a.values())


def combine_dev(lib, **kw):
    a = dict(L_ids=P, L_s=P, n_q=4, k_q=10, slot_id=P, n_used=20000, tab_ids=P, tab_f=P, width=100, gamma=3.0, k_out=100,
             f_out=P, ids_out=P, n_used_dev=P, status=P, stream=NULL)
    a.update(kw)
    return lib.mdir_diffusion_combine_dev(*a.values())


def test_solve_dev_refusals(lib):
    for name in ("L_ids", "L_s", "slot_id", "nbr", "S", "f_out", "ids_out"):
        assert solve_dev(lib, **{name: NULL}) != 0, name
    for bad in (dict(trunc=0), dict(trunc=2049, k_out=100), dict(k_q=0), dict(k_q=1001), dict(k=0), dict(k=256),
                dict(k_out=0), dict(k_out=1001), dict(n_q=-1), dict(n_used=-1), dict(alpha=1.0), dict(iters=0), dict(rtol=-1.0),
                dict(gamma=0.0)):
        assert solve_dev(lib, **bad) != 0, bad
        assert lib.mdir_last_error()
    # every argument valid but the workspace: refused on the host as well (n_q = 4 needs 4 CTAs' ELL)
    assert solve_dev(lib, ws_bytes=lib.mdir_diffusion_solve_workspace_bytes(4, 1000, 50) - 1) != 0
    assert solve_dev(lib, ws=NULL, ws_bytes=1 << 30) != 0
    assert b"ws" in lib.mdir_last_error()


def test_combine_dev_refusals(lib):
    for name in ("L_ids", "L_s", "slot_id", "tab_ids", "tab_f", "f_out", "ids_out"):
        assert combine_dev(lib, **{name: NULL}) != 0, name
    for bad in (dict(k_q=0), dict(k_q=129, width=10), dict(width=0), dict(width=1025, k_q=1), dict(k_q=82, width=100),
                dict(k_out=0), dict(k_out=8193), dict(n_q=-1), dict(n_used=-1), dict(gamma=0.0)):
        assert combine_dev(lib, **bad) != 0, bad
        assert lib.mdir_last_error()


def test_zero_queries_launch_nothing(lib):
    """n_q = 0 is a valid empty batch: success without touching the device, optional pointers NULL or not."""
    assert solve_dev(lib, n_q=0, ws=NULL) == 0 and solve_dev(lib, n_q=0, n_used_dev=NULL, status=NULL) == 0
    assert combine_dev(lib, n_q=0) == 0 and combine_dev(lib, n_q=0, n_used_dev=NULL, status=NULL) == 0


def test_serving_parameter_refusals_without_gpu():
    import mdir_b200
    from mdir_b200 import diffusion as dif
    E = mdir_b200.MdirError
    g = dif.Diffusion.__new__(dif.Diffusion)
    tab = dif.DiffusionTable.__new__(dif.DiffusionTable)
    tab.width = 100
    with pytest.raises(E, match="Diffusion or a DiffusionTable"):
        mdir_b200.GraphedDiffusion(object(), 70)
    with pytest.raises(TypeError, match="trunc"):
        mdir_b200.GraphedDiffusion(tab, 70, trunc=1000)                   # a table's search has no shortlist
    with pytest.raises(TypeError, match="beta"):
        mdir_b200.GraphedDiffusion(g, 70, beta=1)
    for n_q in (0, 129):
        with pytest.raises(E, match="n_q"):
            mdir_b200.GraphedDiffusion(g, n_q)
    for bad in (dict(k=0), dict(trunc=2049), dict(k=1001), dict(k_q=0), dict(alpha=1.0), dict(iters=0), dict(rtol=-1.0)):
        with pytest.raises(E):
            mdir_b200.GraphedDiffusion(g, 70, **bad)
    for bad in (dict(k_q=0), dict(k_q=82), dict(k=8193)):
        with pytest.raises(E):
            mdir_b200.GraphedDiffusion(tab, 70, **bad)
    with pytest.raises(E, match="depth"):
        mdir_b200.DiffusionPipeline(g, 70, depth=0)
    assert dif._serving_params(tab, {}) == {"k_q": 10}
    assert dif._serving_params(g, {"k_q": 5}) == dict(trunc=1000, k_q=5, alpha=0.99, iters=20, rtol=1e-6)
