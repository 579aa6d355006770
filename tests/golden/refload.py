"""Loader for the UNMODIFIED reference modules (only usable with TSD_REFERENCE_ROOT set to a checkout of
cfkr-dev/OpenCV-Traffic-Sign-Detector, which is not part of this repository).

Test infrastructure: used by tests/golden/make_golden.py to generate golden vectors and by the
optional `-m "not gpu"` tests that re-validate the oracle against the live reference when the
reference tree is present.  Nothing on the product path imports this file.

The two reference packages both call their modules `source` / `constants`
(DET = "Deteción de Objetos", REC = "Reconocimiento de Objetos"), so they are loaded under
distinct names with the matching `constants` pre-seeded in sys.modules (SURVEY.md App. C).
REC/source.py:25 imports matplotlib, which is not installed -> a stub package is injected.
"""
import importlib.util
import os
import sys
import types

REF_ROOT = os.environ.get("TSD_REFERENCE_ROOT", "")
DET_DIR = os.path.join(REF_ROOT, "Deteción de Objetos")
REC_DIR = os.path.join(REF_ROOT, "Reconocimiento de Objetos")


def reference_available():
    return bool(REF_ROOT) and os.path.isfile(os.path.join(DET_DIR, "source.py")) and os.path.isfile(os.path.join(REC_DIR, "source.py"))


def _stub_matplotlib():
    if "matplotlib" in sys.modules:
        return
    try:
        import matplotlib  # noqa: F401
        return
    except Exception:
        pass

    class _Any(types.ModuleType):
        def __getattr__(self, name):
            if name.startswith("__"):
                raise AttributeError(name)
            return lambda *a, **k: None

    mpl = _Any("matplotlib")
    mpl.__path__ = []
    sys.modules["matplotlib"] = mpl
    sys.modules["matplotlib.pyplot"] = _Any("matplotlib.pyplot")


def _load(pkg_dir, alias):
    _stub_matplotlib()
    cspec = importlib.util.spec_from_file_location(alias + "_constants", os.path.join(pkg_dir, "constants.py"))
    cmod = importlib.util.module_from_spec(cspec)
    cspec.loader.exec_module(cmod)
    saved = sys.modules.get("constants")
    sys.modules["constants"] = cmod
    try:
        sspec = importlib.util.spec_from_file_location(alias + "_source", os.path.join(pkg_dir, "source.py"))
        smod = importlib.util.module_from_spec(sspec)
        sspec.loader.exec_module(smod)
    finally:
        if saved is not None:
            sys.modules["constants"] = saved
        else:
            sys.modules.pop("constants", None)
    return smod, cmod


_cache = {}


def load_det():
    """-> (source module, constants module) of the detection package."""
    if "det" not in _cache:
        _cache["det"] = _load(DET_DIR, "refdet")
    return _cache["det"]


def load_rec():
    """-> (source module, constants module) of the recognition package."""
    if "rec" not in _cache:
        _cache["rec"] = _load(REC_DIR, "refrec")
    return _cache["rec"]
