"""Import the LIVE reference (the jenicek/mdir source tree) from the first of: $MDIR_REF_ROOT, oracle/_ref/, and the
verbatim copy that ``baseline/stage_ref.py`` places under baseline/_ref/ (both directories git-ignored: reference
sources never enter this repository).  Without any of them the tests that need the reference skip.

TEST INFRASTRUCTURE ONLY: used by ``oracle/make_golden.py`` (golden vectors committed under tests/golden/),
by the integration tests (validate() un-patched vs after mdir_b200.install()) and by bench.py's CPU-baseline
legs.  Never imported by the product package.  Recipe: SURVEY.md App. B (stub two absent off-path modules,
alias a Pillow constant that Pillow 12 dropped).
"""
import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _find_root():
    cands = (os.environ.get("MDIR_REF_ROOT"), os.path.join(_REPO, "oracle", "_ref"), os.path.join(_REPO, "baseline", "_ref"))
    for cand in cands:
        if cand and os.path.isdir(os.path.join(cand, "mdir")):
            return cand
    return cands[1]


REF_ROOT = _find_root()


def available():
    return os.path.isdir(os.path.join(REF_ROOT, "mdir"))


def import_reference():
    """Returns the imported ``mdir`` package (cirtorch is importable afterwards)."""
    if not available():
        raise RuntimeError("reference tree not found (set MDIR_REF_ROOT, or place it under oracle/_ref or baseline/_ref)")
    sys.dont_write_bytecode = True
    if "h5py" not in sys.modules:
        sys.modules["h5py"] = types.ModuleType("h5py")          # daan file readers only
    if "matplotlib" not in sys.modules:
        mpl = types.ModuleType("matplotlib")
        mpl.use = lambda *a, **k: None
        mpl.rcParams = {"font.size": 10.0}
        plt = types.ModuleType("matplotlib.pyplot")
        mpl.pyplot = plt
        sys.modules["matplotlib"] = mpl
        sys.modules["matplotlib.pyplot"] = plt
    from PIL import Image
    if not hasattr(Image, "ANTIALIAS"):
        Image.ANTIALIAS = Image.LANCZOS
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import mdir  # noqa: F401  (side effects: torch threads=3, cv2 threads=1)
    return mdir
