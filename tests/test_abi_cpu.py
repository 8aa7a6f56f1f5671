"""CPU tests of the boundary: the C-ABI library builds/loads, exports every symbol the header
declares, the Python mirror exposes the reference's names, and the product path fails LOUDLY
without a GPU (no CPU fallback, no route through oracle/)."""
import os
import re
import subprocess
import sys

import pytest
import torch

from tests.util import ROOT


def test_library_exports_every_declared_symbol(lib):
    from anyloc_b200 import _lib
    header = open(os.path.join(ROOT, "include", "anyloc_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(anyloc_[a-z0-9_]+)\s*\(", header)))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/anyloc_b200.h but not exported"
    assert set(declared) == set(_lib.EXPORTS), set(declared) ^ set(_lib.EXPORTS)
    assert lib.anyloc_version() >= 100


def test_library_contains_sm100a_code(lib):
    from anyloc_b200 import _lib
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def test_mirror_api_surface():
    from anyloc_b200 import utilities as u
    for name in ("VLAD", "DinoV2ExtractFeatures", "get_top_k_recall", "seed_everything", "reduce_pca",
                 "CustomDataset", "to_np", "to_pil_list", "pad_img", "concat_desc_dists_clusters"):
        assert hasattr(u, name)
    import inspect
    sig = inspect.signature(u.VLAD.__init__)
    assert list(sig.parameters)[1:] == ["num_clusters", "desc_dim", "intra_norm", "norm_descs", "dist_mode",
                                        "vlad_mode", "soft_temp", "cache_dir"]          # utilities.py:657-662
    assert sig.parameters["dist_mode"].default == "cosine" and sig.parameters["vlad_mode"].default == "hard"
    sig = inspect.signature(u.DinoV2ExtractFeatures.__init__)
    assert list(sig.parameters)[1:7] == ["dino_model", "layer", "facet", "use_cls", "norm_descs", "device"]
    sig = inspect.signature(u.get_top_k_recall)
    assert list(sig.parameters) == ["top_k", "db", "qu", "gt_pos", "method", "norm_descs", "use_gpu",
                                    "use_percentage", "sub_sample_db", "sub_sample_qu"]  # utilities.py:390-394
    for m in ("fit", "fit_and_generate", "generate", "generate_multi", "generate_res_vec",
              "generate_multi_res_vec", "can_use_cache_vlad", "can_use_cache_ids"):
        assert callable(getattr(u.VLAD, m))


def test_dropin_shim_resolves_utilities():
    code = ("import sys; sys.path.insert(0, %r); import utilities as U; "
            "print(U.VLAD.__module__, U.DinoV2ExtractFeatures.__module__, U.get_top_k_recall.__module__)"
            % os.path.join(ROOT, "anyloc_b200", "dropin"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd="/tmp")
    assert out.returncode == 0, out.stderr
    assert out.stdout.strip().splitlines()[-1] == "anyloc_b200.utilities " * 2 + "anyloc_b200.utilities"


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_fails_loudly_without_gpu(lib):
    from anyloc_b200 import utilities as u, _lib
    v = u.VLAD(4)
    v.kmeans, v.c_centers, v.desc_dim = u._KMeans(4, mode="cosine"), torch.randn(4, 8), 8
    with pytest.raises(_lib.AnylocError):
        v.generate(torch.randn(10, 8))
    with pytest.raises(_lib.AnylocError):
        u.get_top_k_recall([1], torch.randn(5, 8), torch.randn(2, 8), [[0], [1]])
    with pytest.raises(_lib.AnylocError):
        u.DinoV2ExtractFeatures("dinov2_vits14", 3, "value", device="cuda")
    assert lib.anyloc_device_info(None, None) < 0 and "no CUDA device" in _lib.last_error()


def test_product_never_imports_oracle():
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "anyloc_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", src, re.M) or "/root/reference" in src.replace(
                        "/root/reference/utilities.py", "").replace("/root/reference/", ""):
                    bad.append(f)
    assert not bad, bad


def test_cache_predicates_and_fit_errors(tmp_path):
    from anyloc_b200 import utilities as u
    v = u.VLAD(3, cache_dir=str(tmp_path / "cache"))
    assert (tmp_path / "cache").is_dir() and not v.can_use_cache_vlad() and not v.can_use_cache_ids(["a"])
    torch.save(torch.randn(3, 16), tmp_path / "cache" / "c_centers.pt")
    assert v.can_use_cache_vlad() and not v.can_use_cache_ids("a")
    torch.save(torch.zeros(1), tmp_path / "cache" / "a_r.pt")
    assert v.can_use_cache_ids("a", only_residuals=True) and not v.can_use_cache_ids("a")
    torch.save(torch.zeros(1), tmp_path / "cache" / "a_l.pt")
    assert v.can_use_cache_ids(["a"])
    v.fit(None)                                              # vocabulary restored from cache, no GPU needed
    assert v.desc_dim == 16 and v.c_centers.shape == (3, 16)
    with pytest.raises(ValueError):
        u.VLAD(3).fit(None)


def test_host_helpers_match_reference():
    """the pass-through helpers of utilities.py (:99-129 to_pil_list, :474-500 pad_img, :590-619
    concat_desc_dists_clusters) against the reference's outputs (tests/golden/reference_checks.npz)"""
    import numpy as np
    from anyloc_b200 import utilities as u
    from tests.util import host_helper_inputs, load_cases
    g = load_cases("reference_checks.npz")["helpers"]
    c, x, img, batches = host_helper_inputs()
    assert torch.equal(torch.from_numpy(g["concat"]), u.concat_desc_dists_clusters(c, x))
    assert np.array_equal(g["pad"], u.pad_img(img, 2, [255, 0, 3]))
    for b, batch in enumerate(batches):
        ref = [g[k] for k in sorted(k for k in g if k.startswith(f"pil{b}_"))]
        ours = u.to_pil_list(batch)
        assert len(ref) == len(ours) and all(np.array_equal(p, np.asarray(q)) for p, q in zip(ref, ours))
