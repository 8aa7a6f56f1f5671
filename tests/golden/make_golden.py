"""Generates the committed golden vectors under tests/golden/ by running the
REFERENCE'S OWN CODE (/root/reference/utilities.py, imported verbatim through
oracle/reference_import.py) on seeded inputs.  Run in the build container only:

    python tests/golden/make_golden.py

Third-party arithmetic the reference does not vendor (dinov2 hub model,
fast_pytorch_kmeans, faiss) is supplied by the restatements in oracle/ -- see
oracle/__init__.py for what is and is not pinned.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import reference_import as ri           # noqa: E402
from oracle import anyloc_oracle as ao              # noqa: E402
from oracle import dinov2_restated as dr            # noqa: E402
from oracle import fpk_restated as fpk              # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
ref = ri.load_reference_utilities()


def ref_vlad(K, centers, **kw):
    v = ref.VLAD(K, **kw)
    v.kmeans = fpk.KMeans(K, mode=v.mode)
    v.kmeans.centroids = centers
    v.c_centers = centers
    v.desc_dim = centers.shape[1]
    return v


def make_vlad():
    cases = {}
    g = torch.Generator().manual_seed(123)
    specs = [
        # name, N, D, K, kind, kwargs
        ("clustered_n300_d64_k8", 300, 64, 8, "clustered", {}),
        ("random_n257_d96_k5", 257, 96, 5, "random", {}),
        ("random_n64_d32_k1", 64, 32, 1, "random", {}),
        ("nointra_n100_d48_k4", 100, 48, 4, "clustered", {"intra_norm": False}),
        ("nonorm_n100_d48_k4", 100, 48, 4, "random_unnorm", {"norm_descs": False}),
        ("euclid_n120_d40_k6", 120, 40, 6, "random_unnorm", {"dist_mode": "euclidean"}),
        ("emptyclusters_n10_d32_k16", 10, 32, 16, "clustered", {}),
        ("ties_zero_n40_d32_k4", 40, 32, 4, "ties", {}),
    ]
    for name, N, D, K, kind, kw in specs:
        if kind == "clustered":
            x, c, _ = ao.clustered_features(N, D, K, seed=len(name))
        elif kind == "random":
            x = torch.nn.functional.normalize(torch.randn(N, D, generator=g), dim=1)
            c = 0.7 * torch.nn.functional.normalize(torch.randn(K, D, generator=g), dim=1)
        elif kind == "random_unnorm":
            x = torch.randn(N, D, generator=g) * (0.5 + torch.rand(N, 1, generator=g))
            c = torch.randn(K, D, generator=g) * 0.8
        elif kind == "ties":
            x, c, _ = ao.clustered_features(N, D, K, seed=5)
            c[2] = c[1]                      # duplicate centre -> exact tie, lowest index wins
            x[3] = 0.0                       # all-zero descriptor -> label 0
            x[7] = 0.0
        v = ref_vlad(K, c, **kw)
        out = v.generate(x)
        labels = v.kmeans.predict(x)
        cases[name] = dict(x=x.numpy(), centers=c.numpy(), out=out.numpy(),
                           labels=labels.numpy().astype(np.int64),
                           kw=np.array(repr(kw)))
    # generate_multi on a batch and on a ragged list
    x, c, _ = ao.clustered_features(4 * 50, 32, 6, seed=9)
    v = ref_vlad(6, c)
    xb = x.reshape(4, 50, 32)
    cases["multi_b4_n50_d32_k6"] = dict(x=xb.numpy(), centers=c.numpy(),
                                        out=v.generate_multi(xb).numpy(), kw=np.array("{}"))
    flat = {}
    for n, d in cases.items():
        for k, a in d.items():
            flat[f"{n}/{k}"] = a
    np.savez_compressed(os.path.join(OUT, "vlad.npz"), **flat)
    print("vlad.npz", len(cases), "cases")


def make_vlad_soft():
    # the soft branch of VLAD.generate (utilities.py:862-887)
    g = torch.Generator().manual_seed(321)
    cases = {}
    specs = [
        ("soft_t1_n90_d48_k6", 90, 48, 6, "clustered", {"soft_temp": 1.0}),
        ("soft_t20_n130_d64_k8", 130, 64, 8, "clustered", {"soft_temp": 20.0}),
        ("soft_t5_nonorm_n70_d40_k5", 70, 40, 5, "random_unnorm", {"soft_temp": 5.0, "norm_descs": False}),
        ("soft_t3_nointra_n60_d32_k37", 60, 32, 37, "random_unnorm", {"soft_temp": 3.0, "intra_norm": False}),
        ("soft_t10_zero_n33_d36_k3", 33, 36, 3, "zero", {"soft_temp": 10.0}),
    ]
    for name, N, D, K, kind, kw in specs:
        if kind in ("clustered", "zero"):
            x, c, _ = ao.clustered_features(N, D, K, seed=len(name))
            if kind == "zero":
                x[5] = 0.0                   # cos = 0 to every centre -> uniform weights
        else:
            x = torch.randn(N, D, generator=g) * (0.5 + torch.rand(N, 1, generator=g))
            c = torch.randn(K, D, generator=g) * 0.8
        v = ref_vlad(K, c, vlad_mode="soft", **kw)
        cases[name] = dict(x=x.numpy(), centers=c.numpy(), out=v.generate(x).numpy(), kw=np.array(repr(kw)))
    x, c, _ = ao.clustered_features(3 * 40, 32, 4, seed=11)
    v = ref_vlad(4, c, vlad_mode="soft", soft_temp=8.0)
    xb = x.reshape(3, 40, 32)
    cases["multi_soft_t8_b3_n40_d32_k4"] = dict(x=xb.numpy(), centers=c.numpy(), out=v.generate_multi(xb).numpy(),
                                                kw=np.array(repr({"soft_temp": 8.0})))
    flat = {}
    for n, d in cases.items():
        for k, a in d.items():
            flat[f"{n}/{k}"] = a
    np.savez_compressed(os.path.join(OUT, "vlad_soft.npz"), **flat)
    print("vlad_soft.npz", len(cases), "cases")


def make_fit():
    # VLAD.fit (utilities.py:749-791) through the restated fpk KMeans; numpy RNG seeded as the
    # reference does at import / in main (seed_everything -> np.random.seed(42)).
    x, _, _ = ao.clustered_features(400, 24, 5, seed=3, kappa_noise=0.8)
    np.random.seed(42)
    v = ref.VLAD(5)
    v.fit(x)
    np.savez_compressed(os.path.join(OUT, "fit.npz"), x=x.numpy(), centers=v.c_centers.numpy())
    print("fit.npz")


def make_topk():
    g = torch.Generator().manual_seed(7)
    db = torch.randn(60, 80, generator=g)
    qu = db[torch.randperm(60, generator=g)[:9]] + 0.3 * torch.randn(9, 80, generator=g)
    db[11] = db[4]                                   # duplicate rows -> lowest index first
    gt = np.empty(9, dtype=object)
    for i in range(9):
        gt[i] = np.array([(3 * i) % 60, (7 * i + 1) % 60])
    out = {}
    for method in ("cosine", "l2"):
        d, i, r = ref.get_top_k_recall([1, 3, 5], db, qu, gt, method=method)
        out[f"{method}/dist"], out[f"{method}/idx"] = d.numpy(), i.numpy()
        out[f"{method}/recalls"] = np.array([r[k] for k in (1, 3, 5)])
    d, i, r = ref.get_top_k_recall([2], db, qu[0], gt, method="cosine", norm_descs=False,
                                   use_percentage=False)
    out["single/dist"], out["single/idx"] = d.numpy(), i.numpy()
    out["single/recalls"] = np.array([r[2]])
    gt_obj = np.array([g_.tolist() for g_ in gt], dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, "topk.npz"), db=db.numpy(), qu=qu.numpy(), gt=gt_obj, **out)
    print("topk.npz")


def make_extract():
    out = {}
    cfgs = [
        # tag, model, depth_override, layer, H, W
        ("vits14_l9_56x70", "dinov2_vits14", None, 9, 56, 70),
        ("vitg14_d2_l1_42x42", "dinov2_vitg14", 2, 1, 42, 42),
    ]
    for tag, name, depth, layer, H, W in cfgs:
        factory = lambda n, depth=depth: dr.perturb(dr.build(n, seed=0, depth_override=depth), seed=1)
        img = torch.randn(2, 3, H, W, generator=torch.Generator().manual_seed(1234))
        out[f"{tag}/img"] = img.numpy()
        for facet in ("value", "key", "query", "token"):
            with ri.hub_patched(factory):
                ext = ref.DinoV2ExtractFeatures(name, layer, facet, device="cpu")
            feats = ext(img)
            out[f"{tag}/{facet}"] = feats.numpy()
        with ri.hub_patched(factory):
            ext = ref.DinoV2ExtractFeatures(name, layer, "value", use_cls=True, norm_descs=False, device="cpu")
        out[f"{tag}/value_cls_nonorm"] = ext(img).numpy()
    np.savez_compressed(os.path.join(OUT, "extract.npz"), **out)
    print("extract.npz")


def make_preprocess():
    # base_transform (dvgl_benchmark/datasets_ws.py:20-23) + the centre crop of scripts/dino_v2_vlad.py:174-176,
    # run through torchvision itself on PIL images (small sizes: inputs and full outputs are stored).
    import torchvision.transforms as T
    from PIL import Image
    base_transform = T.Compose([T.ToTensor(), T.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
    rng = np.random.default_rng(77)
    out = {}
    for tag, (h, w) in {"a_45x61": (45, 61), "b_30x28": (30, 28), "c_59x43": (59, 43), "d_14x27": (14, 27)}.items():
        img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        img[0, 0] = (0, 255, 128)
        t = base_transform(Image.fromarray(img, "RGB"))
        hn, wn = (h // 14) * 14, (w // 14) * 14
        res = T.CenterCrop((hn, wn))(t)
        out[f"{tag}/img"] = img
        out[f"{tag}/out"] = res.numpy()
    np.savez_compressed(os.path.join(OUT, "preprocess.npz"), **out)
    print("preprocess.npz")
    # with the dataset loader's resize (dvgl_benchmark/datasets_ws.py:233-235, `T.functional.resize(img, self.resize)` on
    # the normalised tensor) / the demo's bicubic down-scaling (demo/anyloc_vlad_generate.py:165-177), by torchvision
    out = {}
    for tag, (h, w), size, mode in (("bilinear_97x131_to_60x80", (97, 131), (60, 80), T.InterpolationMode.BILINEAR),
                                    ("bilinear_40x52_to_60x80", (40, 52), (60, 80), T.InterpolationMode.BILINEAR),
                                    ("bicubic_150x90_to_70x42", (150, 90), (70, 42), T.InterpolationMode.BICUBIC),
                                    ("bicubic_33x47_to_58x83", (33, 47), (58, 83), T.InterpolationMode.BICUBIC)):
        img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        t = T.functional.resize(base_transform(Image.fromarray(img, "RGB")), list(size), interpolation=mode)
        res = T.CenterCrop(((size[0] // 14) * 14, (size[1] // 14) * 14))(t)
        out[f"{tag}/img"] = img
        out[f"{tag}/out"] = res.numpy()
        out[f"{tag}/size"] = np.array(size)
    np.savez_compressed(os.path.join(OUT, "preprocess_resize.npz"), **out)
    print("preprocess_resize.npz")


def make_build_vlads():
    """The reference's UNMODIFIED driver -- `build_vlads` of scripts/dino_v2_vlad.py:124-303 -- over its own
    utilities.py on the synthetic dataset of tests/dropin_harness.py (hard and soft assignment), then its own
    get_top_k_recall.  tests/test_dropin_gpu.py replays the dataset through the shim on the GPU against these."""
    from tests import dropin_harness as H
    script = H.load_script(ref)
    out = {}
    for tag, soft in (("hard", False), ("soft", True)):
        ds = H.SyntheticVprDataset()
        model_factory = lambda name: dr.perturb(dr.build(name, seed=0, depth_override=3), seed=3)
        with ri.hub_patched(model_factory):
            np.random.seed(42)
            largs = H.make_largs(script, "/tmp/_anyloc_golden_cache", "dinov2_vits14", 2, "value", 4, False, soft)
            db, qu = script.build_vlads(largs, ds, verbose=False)
            # the vocabulary the run fitted (same seed -> same k-means): refit outside to record it
            np.random.seed(42)
            v = ref.VLAD(4, vlad_mode="soft" if soft else "hard")
            dino = ref.DinoV2ExtractFeatures("dinov2_vits14", 2, "value", device="cpu")
            from torchvision import transforms as T
            feats = torch.cat([dino(T.CenterCrop((56, 70))(ds[i][0])[None]) for i in range(ds.database_num)])
            v.fit(feats.reshape(-1, feats.shape[-1]))
        assert torch.equal(v.generate_multi(feats), db)
        d, i, rec = ref.get_top_k_recall([1, 2, 3], db, qu, ds.soft_positives_per_query)
        out[f"{tag}/db_vlads"], out[f"{tag}/qu_vlads"] = db.numpy(), qu.numpy()
        out[f"{tag}/c_centers"] = v.c_centers.numpy()
        out[f"{tag}/dist"], out[f"{tag}/idx"] = np.asarray(d), np.asarray(i)
        out[f"{tag}/recalls"] = np.array([rec[1], rec[2], rec[3]])
    np.savez_compressed(os.path.join(OUT, "build_vlads.npz"), **out)
    print("build_vlads.npz")


def make_reference_checks():
    """The reference's VLAD.generate and get_top_k_recall, reduce_pca (both branches) and host helpers (to_pil_list,
    pad_img, concat_desc_dists_clusters) on the seeded inputs of tests/util.py, which the tests regenerate."""
    from tests import util as U
    out = {}
    vlads, db, qu, gt = U.vlad_topk_check_inputs()
    for j, (x, c) in enumerate(vlads):
        out[f"vlad{j}/out"] = ref_vlad(c.shape[0], c).generate(x).numpy()
    d, i, r = ref.get_top_k_recall([1, 4], db, qu, gt)
    out["topk/dist"], out["topk/idx"], out["topk/recalls"] = d.numpy(), i.numpy(), np.array([r[1], r[4]])
    tr, te = U.pca_check_inputs()
    for j, kw in enumerate(U.PCA_CHECK_KWARGS):
        a = ref.reduce_pca(tr.copy(), te.copy(), 8, **kw)
        out[f"pca{j}/train"], out[f"pca{j}/test"] = a[0], a[1]
    c, x, img, batches = U.host_helper_inputs()
    out["helpers/concat"] = ref.concat_desc_dists_clusters(c, x).numpy()
    out["helpers/pad"] = ref.pad_img(img, 2, (255, 0, 3))
    for b, batch in enumerate(batches):
        for j, p in enumerate(ref.to_pil_list(batch)):
            out[f"helpers/pil{b}_{j}"] = np.asarray(p)
    np.savez_compressed(os.path.join(OUT, "reference_checks.npz"), **out)
    print("reference_checks.npz")


def make_dropin():
    """What the reference's unmodified driver (`build_vlads`) leaves in its --cache-vlad-descs directory on the
    synthetic dataset of tests/dropin_harness.py (hard and soft): the file list with each tensor's dtype and shape,
    the vocabulary and assignments in full, the residual files as digests (tests/util.py).  Its descriptors equal
    the uncached run's (build_vlads.npz).  Also the residual tensor of VLAD.generate_multi_res_vec, as a digest."""
    import tempfile
    from tests import dropin_harness as H
    from tests import util as U
    script = H.load_script(ref)
    bv = U.load_cases("build_vlads.npz")
    out = {}
    for tag, soft in (("hard", False), ("soft", True)):
        ds = H.SyntheticVprDataset()
        with tempfile.TemporaryDirectory() as tmp, ri.hub_patched(H.hub_model):
            np.random.seed(42)
            largs = H.make_largs(script, tmp, H.MODEL, H.LAYER, "value", H.K, True, soft)
            db, qu = script.build_vlads(largs, ds, verbose=False)
            assert np.array_equal(db.numpy(), bv[tag]["db_vlads"]) and np.array_equal(qu.numpy(), bv[tag]["qu_vlads"])
            cdir = H.cache_subdir(tmp)
            meta = []
            for dirpath, _, files in os.walk(cdir):
                for f in files:
                    rel = os.path.relpath(os.path.join(dirpath, f), cdir)
                    t = torch.load(os.path.join(cdir, rel))
                    meta.append(f"{rel}|{t.dtype}|{tuple(t.shape)}")
                    if rel == "c_centers.pt":
                        out[f"{tag}/c_centers"] = t.numpy()
                    elif rel.endswith("_r.pt"):
                        for k, v in U.digest(t.numpy()).items():
                            out[f"{tag}/{rel[:-5]}_r_{k}"] = v
                    else:
                        out[f"{tag}/{rel[:-3]}"] = t.numpy()
            out[f"{tag}/files"] = np.array(sorted(meta))
    x, centers = H.residual_api_inputs()
    with tempfile.TemporaryDirectory() as tmp:
        torch.save(centers, os.path.join(tmp, "c_centers.pt"))
        vr = ref.VLAD(5, cache_dir=tmp)
        vr.fit(None)
        for k, v in U.digest(vr.generate_multi_res_vec(x).numpy()).items():
            out[f"residual_api/{k}"] = v
    np.savez_compressed(os.path.join(OUT, "dropin.npz"), **out)
    print("dropin.npz")


if __name__ == "__main__":
    makers = {"vlad": make_vlad, "vlad_soft": make_vlad_soft, "fit": make_fit, "topk": make_topk,
              "extract": make_extract, "preprocess": make_preprocess, "build_vlads": make_build_vlads,
              "reference_checks": make_reference_checks, "dropin": make_dropin}
    for name in (sys.argv[1:] or list(makers)):      # `make_golden.py vlad_soft` regenerates one file
        makers[name]()
