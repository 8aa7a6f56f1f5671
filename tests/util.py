"""Shared helpers for the parity tests (the oracle is the checker, never the thing under test)."""
import ast
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def load_cases(fname):
    z = np.load(os.path.join(GOLDEN, fname), allow_pickle=False)
    cases = {}
    for key in z.files:
        if "/" in key:
            name, field = key.split("/", 1)
            cases.setdefault(name, {})[field] = z[key]
        else:
            cases.setdefault("", {})[key] = z[key]
    return cases


def case_kwargs(case):
    return ast.literal_eval(str(case["kw"])) if "kw" in case else {}


def rel_inf(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def digest(a, n=64):
    """Pins an array too large to store: shape, float64 sum and sum of squares, and `n` entries at seeded positions."""
    a = np.asarray(a)
    flat = a.reshape(-1)
    pos = np.random.default_rng(0).choice(flat.size, min(n, flat.size), replace=False)
    return dict(shape=np.array(a.shape), sums=np.array([flat.astype(np.float64).sum(),
                                                         np.square(flat.astype(np.float64)).sum()]),
                pos=pos, vals=flat[pos])


def matches_digest(a, d, tol=0.0):
    """`a` against digest(b): bit for bit when tol == 0, else the sampled entries within tol of their largest
    magnitude and the sum of squares within relative tol"""
    a = np.asarray(a)
    flat = a.reshape(-1).astype(np.float64)
    if tuple(a.shape) != tuple(d["shape"]):
        return False
    sums = np.array([flat.sum(), np.square(flat).sum()])
    if tol == 0:
        return np.array_equal(flat[d["pos"]], d["vals"]) and np.array_equal(sums, d["sums"])
    return (np.abs(flat[d["pos"]] - d["vals"]).max() <= tol * np.abs(d["vals"]).max() and
            abs(sums[1] - d["sums"][1]) <= tol * d["sums"][1])


def vlad_topk_check_inputs():
    """Seeded inputs of the VLAD.generate / get_top_k_recall comparison with the reference
    (tests/golden/reference_checks.npz): [(x, centers)] for three shapes, then db, qu, gt."""
    g = torch.Generator().manual_seed(5)
    vlads = []
    for (N, D, K) in [(200, 64, 8), (529, 128, 32), (17, 32, 3)]:
        x = torch.nn.functional.normalize(torch.randn(N, D, generator=g), dim=1)
        vlads.append((x, 0.6 * torch.randn(K, D, generator=g)))
    db, qu = torch.randn(40, 64, generator=g), torch.randn(6, 64, generator=g)
    gt = np.empty(6, dtype=object)
    for i in range(6):
        gt[i] = np.array([i, i + 1])
    return vlads, db, qu, gt


def pca_check_inputs():
    g = np.random.default_rng(0)
    tr = (g.standard_normal((200, 24)) * (0.8 ** np.arange(24))).astype(np.float32)
    te = (g.standard_normal((31, 24)) * (0.8 ** np.arange(24))).astype(np.float32)
    return tr, te


PCA_CHECK_KWARGS = (dict(whitening=False), dict(whitening=True), dict(low_factor=0.25))


def host_helper_inputs():
    """-> centres, descriptors (concat_desc_dists_clusters), a uint8 image (pad_img), two batches (to_pil_list)"""
    g = torch.Generator().manual_seed(0)
    c, x = torch.randn(5, 16, generator=g), torch.randn(9, 16, generator=g)
    img = (np.random.default_rng(0).random((10, 12, 3)) * 255).astype(np.uint8)
    return c, x, img, (torch.rand(2, 3, 8, 9, generator=g), torch.rand(8, 9, 3, generator=g))


def make_vlad(u, K, centers, **kw):
    """product VLAD object with a given vocabulary (what `fit` from a c_centers.pt cache yields)."""
    v = u.VLAD(K, **kw)
    v.kmeans = u._KMeans(K, mode=v.mode)
    v.kmeans.centroids = torch.as_tensor(centers)
    v.c_centers = torch.as_tensor(centers)
    v.desc_dim = centers.shape[1]
    return v
