"""Import the UNMODIFIED reference modules from an upstream HTR-VT source tree (set HTRVT_REFERENCE to it).

TEST INFRASTRUCTURE ONLY: oracle/make_golden.py uses it to regenerate tests/golden/.  The tree is not part of this
repository, so nothing in the test suite, smoke() or bench.py may call this.
"""
import importlib
import os
import sys

REF_ROOT = os.environ.get("HTRVT_REFERENCE", "/root/reference")
_STUB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "timm_stub")


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "model_v1", "model"))


def load_variant(variant: str = "model_v1"):
    """Return (HTR_VT module, utils.utils module) of a reference variant directory.

    The reference uses top-level package names `model` / `utils` inside each variant
    directory (model_v1/train.py:9-13), so modules from a previously loaded variant are purged.
    """
    if not available():
        raise RuntimeError("reference tree not present at %s" % REF_ROOT)
    for name in [m for m in sys.modules if m == "model" or m.startswith("model.")
                 or m == "utils" or m.startswith("utils.")]:
        del sys.modules[name]
    vdir = os.path.join(REF_ROOT, variant)
    for p in (_STUB, vdir):
        if p in sys.path:
            sys.path.remove(p)
    sys.path.insert(0, _STUB)
    sys.path.insert(0, vdir)
    try:
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            htr = importlib.import_module("model.HTR_VT")
            utl = importlib.import_module("utils.utils")
    finally:
        sys.path.remove(vdir)
    return htr, utl
