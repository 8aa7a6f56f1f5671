"""TEST INFRASTRUCTURE -- import the reference's own /root/reference/dino_extractor.py VERBATIM (nothing is
copied into this repo), for tests/golden/make_golden_dino_v1.py.  Build container only: nothing on the GPU box
may call this.

dino_extractor.py imports `timm` (only used to fetch timm checkpoints; not installed here, so a stub stands in)
and `from utilities import to_np`, which must resolve to the REFERENCE's utilities (imported behind the oracle
stubs of reference_import.py) while the module executes; whatever `utilities` was before (e.g. the product's
drop-in shim) is restored afterwards."""
import importlib.util
import os
import sys
import types

from oracle import reference_import as ri

_cached = None
_MISSING = object()


def available() -> bool:
    return os.path.isfile(os.path.join(ri.REFERENCE_ROOT, "dino_extractor.py")) and ri.available()


def load_reference_dino_extractor():
    """-> the module object of /root/reference/dino_extractor.py (private name `_anyloc_reference_dino_extractor`)"""
    global _cached
    if _cached is not None:
        return _cached
    if not available():
        raise RuntimeError("reference tree not present (only in the build container)")
    ref_utils = ri.load_reference_utilities()
    if "timm" not in sys.modules:
        try:
            import timm  # noqa: F401
        except ImportError:
            sys.modules["timm"] = types.ModuleType("timm")
    saved = sys.modules.get("utilities", _MISSING)
    sys.modules["utilities"] = ref_utils
    try:
        spec = importlib.util.spec_from_file_location(
            "_anyloc_reference_dino_extractor", os.path.join(ri.REFERENCE_ROOT, "dino_extractor.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        if saved is _MISSING:
            sys.modules.pop("utilities", None)
        else:
            sys.modules["utilities"] = saved
    _cached = mod
    return mod
