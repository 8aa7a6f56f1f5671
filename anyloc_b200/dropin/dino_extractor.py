"""`dino_extractor` shim: put this directory FIRST on PYTHONPATH (before the AnyLoc checkout) and the
reference's DINOv1 scripts (`from dino_extractor import ViTExtractor`, e.g. scripts/dino_vlad.py) run their
feature extraction on anyloc_b200 unchanged."""
import os as _os
import sys as _sys

_repo = _os.path.dirname(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))))
if _repo not in _sys.path:
    _sys.path.insert(0, _repo)

from anyloc_b200.dino_v1 import ViTExtractor  # noqa: F401,E402
