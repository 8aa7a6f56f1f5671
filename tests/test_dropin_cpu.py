"""SURVEY.md T10 -- the drop-in claim, tested on the host: the calling pattern of the reference's driver `build_vlads`
(scripts/dino_v2_vlad.py:124-303, restated in tests/dropin_harness.py) runs on the synthetic dataset with this repo's
shim (anyloc_b200/dropin/utilities.py) answering it, and the database / query VLADs, the recalls and the cache files
must agree with what the reference's unmodified driver produced over its own utilities.py (tests/golden/build_vlads.npz
and dropin.npz, made by tests/golden/make_golden.py).  There is no GPU in this tier, so the product's device seams are
replaced by tests/cpu_double.py: what is under test is the HOST logic the driver reaches (constructor arguments,
batch-1 calling pattern, `.cpu()` hand-overs, `vlad.fit(None)` from a cached vocabulary,
`generate_multi(full_db, names)`, `generate_multi([None] * n, names)` on a populated cache, `get_top_k_recall`).  The
kernels behind the seams are checked against the same vectors by the `-m gpu` suite (tests/test_dropin_gpu.py)."""
import os
import sys

import numpy as np
import pytest
import torch
from torch.nn import functional as F

from oracle import anyloc_oracle as ao
from tests import dropin_harness as H
from tests.cpu_double import cpu_double
from tests.util import ROOT, load_cases, matches_digest

MODEL, LAYER, K = H.MODEL, H.LAYER, H.K


@pytest.fixture(scope="module")
def ds():
    return H.SyntheticVprDataset()


@pytest.fixture(scope="module")
def shim():
    sys.path.insert(0, os.path.join(ROOT, "anyloc_b200", "dropin"))
    try:
        import importlib
        spec = importlib.util.spec_from_file_location("_anyloc_shim_utilities",
                                                      os.path.join(ROOT, "anyloc_b200", "dropin", "utilities.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    finally:
        sys.path.pop(0)


def run_shim(shim, ds, cache_dir, cache=False, soft=False):
    with cpu_double(lambda name: H.hub_model(name).state_dict()):
        np.random.seed(42)
        return H.run_driver(shim, ds, cache_dir, cache=cache, soft=soft)


def close(a, b, tol=1e-5):
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    return float((a - b).abs().max() / b.abs().max()) < tol


def reference_run(soft):
    """the reference driver's descriptors on this dataset (uncached and cached runs are identical)"""
    g = load_cases("build_vlads.npz")["soft" if soft else "hard"]
    return torch.from_numpy(g["db_vlads"]), torch.from_numpy(g["qu_vlads"]), g


def cache_files(cdir):
    """-> {relative path: "dtype|shape"} of the tensors under a driver cache directory"""
    out = {}
    for dirpath, _, files in os.walk(cdir):
        for f in files:
            t = torch.load(os.path.join(dirpath, f))
            out[os.path.relpath(os.path.join(dirpath, f), cdir)] = f"{t.dtype}|{tuple(t.shape)}"
    return out


def write_reference_cache(ds, cdir, soft):
    """The cache directory the reference's driver leaves (dropin.npz): vocabulary and assignments as it wrote them;
    the residual files, which are not stored, recomputed with the reference's arithmetic (normalised batch-1 features
    minus the centres) and checked against the digests of the reference's own files."""
    g = load_cases("dropin.npz")["soft" if soft else "hard"]
    files = dict(m.split("|", 1) for m in g["files"].tolist())
    centers = torch.from_numpy(g["c_centers"])
    os.makedirs(os.path.join(cdir, "synth"))
    torch.save(centers, os.path.join(cdir, "c_centers.pt"))
    model = H.hub_model(MODEL)
    for i in range(len(ds)):
        name = ds.get_image_relpaths(i)
        img = ds[i][0]
        feats = ao.extract_features(model, img[None, :, 2:58, 2:72], LAYER, "value")[0]   # T.CenterCrop((56, 70))
        resid = F.normalize(feats)[:, None, :] - centers[None, :, :]
        digest = {k[len(name) + 3:]: v for k, v in g.items() if k.startswith(name + "_r_")}
        assert matches_digest(resid.numpy(), digest, tol=1e-5), name      # ViT features: bit for bit on one CPU only
        torch.save(resid, os.path.join(cdir, name + "_r.pt"))
        sfx = "s" if soft else "l"
        torch.save(torch.from_numpy(g[f"{name}_{sfx}"]), os.path.join(cdir, f"{name}_{sfx}.pt"))
    assert cache_files(cdir) == files
    return files


@pytest.mark.parametrize("soft", [False, True])
def test_driver_loop_matches_reference_run(shim, ds, tmp_path, soft):
    db_r, qu_r, g = reference_run(soft)
    db_s, qu_s = run_shim(shim, ds, str(tmp_path / "shim"), soft=soft)
    assert db_s.shape == db_r.shape == (ds.database_num, K * 384) and qu_s.shape == qu_r.shape
    assert not db_s.is_cuda and db_s.dtype == torch.float32
    assert close(db_s, db_r) and close(qu_s, qu_r)
    top_k = [1, 2, 3]
    with cpu_double():
        d_s, i_s, rec_s = shim.get_top_k_recall(top_k, db_s, qu_s, ds.soft_positives_per_query)
    assert np.array_equal(np.asarray(i_s), g["idx"]) and rec_s == dict(zip(top_k, g["recalls"].tolist()))
    assert rec_s[1] == 1.0
    assert np.allclose(np.asarray(d_s), g["dist"], atol=1e-5)


@pytest.mark.parametrize("soft", [False, True])
def test_cache_directories_are_interchangeable(shim, ds, tmp_path, soft):
    """--cache-vlad-descs (scripts/dino_v2_vlad.py:147-153): (1) a directory as the REFERENCE populates it
    (c_centers.pt, <id>_r.pt, <id>_l.pt | _s.pt) serves the shim, which then never touches the features
    (`[None] * n`, :224-228); (2) the shim's own cache run writes the vocabulary + assignments in the reference's
    format: the same files, dtypes and shapes, the same assignments, so the reference reads them as its own."""
    db_r, qu_r, _ = reference_run(soft)
    ref_dir = str(tmp_path / "cache_ref")
    cdir = H.cache_subdir(ref_dir)
    ref_files = write_reference_cache(ds, cdir, soft)
    sfx = "s" if soft else "l"

    calls = {"n": 0}
    orig = shim.DinoV2ExtractFeatures.__call__

    def counting(self, img):
        calls["n"] += 1
        return orig(self, img)
    shim.DinoV2ExtractFeatures.__call__ = counting
    try:
        db_s, qu_s = run_shim(shim, ds, ref_dir, cache=True, soft=soft)       # reference-populated cache
    finally:
        shim.DinoV2ExtractFeatures.__call__ = orig
    assert calls["n"] == 0, "a complete cache must not trigger any forward pass"
    assert close(db_s, db_r) and close(qu_s, qu_r)

    own = str(tmp_path / "cache_own")
    db_1, qu_1 = run_shim(shim, ds, own, cache=True, soft=soft)               # populates: vocabulary + assignments
    odir = H.cache_subdir(own)
    assert os.path.isfile(os.path.join(odir, "c_centers.pt"))
    lab = torch.load(os.path.join(odir, "synth", f"img_0000.jpg_{sfx}.pt"))
    ref_lab = torch.load(os.path.join(cdir, "synth", f"img_0000.jpg_{sfx}.pt"))
    assert lab.dtype == ref_lab.dtype and lab.shape == ref_lab.shape
    assert torch.equal(lab, ref_lab) if not soft else torch.allclose(lab, ref_lab, atol=1e-6)
    assert not os.path.isfile(os.path.join(odir, "synth", "img_0000.jpg_r.pt")), "the 100 MB/image residual cache is opt-in"
    db_2, qu_2 = run_shim(shim, ds, own, cache=True, soft=soft)               # second run: cached vocabulary + assignments
    assert close(db_1, db_r) and close(db_2, db_r) and close(qu_2, qu_r)
    # what the reference reads back from the shim's directory is what it wrote itself (it recomputes the residuals)
    assert cache_files(odir) == {k: v for k, v in ref_files.items() if not k.endswith("_r.pt")}
    assert torch.allclose(torch.load(os.path.join(odir, "c_centers.pt")), torch.load(os.path.join(cdir, "c_centers.pt")),
                          atol=1e-6)
    for i in range(len(ds)):
        name = ds.get_image_relpaths(i)
        a, b = torch.load(os.path.join(odir, f"{name}_{sfx}.pt")), torch.load(os.path.join(cdir, f"{name}_{sfx}.pt"))
        assert torch.equal(a, b) if not soft else torch.allclose(a, b, atol=1e-6)


def test_residual_tensor_api(shim, tmp_path):
    """VLAD.generate_res_vec / generate_multi_res_vec (utilities.py:928-1008) incl. the `<id>_r.pt` round trip: the
    residual tensor equals the reference's (digest in tests/golden/dropin.npz); the cache file is the plain tensor
    the reference's generate_res_vec loads."""
    x, centers = H.residual_api_inputs()
    torch.save(centers, str(tmp_path / "c_centers.pt"))
    with cpu_double():
        vs = shim.VLAD(5, cache_dir=str(tmp_path))
        vs.fit(None)
        r_s = vs.generate_multi_res_vec(x)
        r_1 = vs.generate_res_vec(x[0].numpy(), "a/b")               # writes a/b_r.pt like the reference
    assert r_s.shape == (2, 40, 5, 64) and matches_digest(r_s.numpy(), load_cases("dropin.npz")["residual_api"])
    cached = torch.load(str(tmp_path / "a" / "b_r.pt"))
    assert type(cached) is torch.Tensor and torch.equal(cached, r_1) and torch.equal(r_1, r_s[0])
    assert vs.can_use_cache_ids(["a/b"], only_residuals=True) and not vs.can_use_cache_ids(["a/b"])
