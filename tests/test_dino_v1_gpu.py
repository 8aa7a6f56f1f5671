"""GPU parity of the DINOv1 ViTExtractor (anyloc_b200.dino_v1) against the reference's own outputs
(tests/golden/dino_v1.npz) and the CPU oracle (oracle/dino_v1_restated.py), of anyloc_log_bin against the oracle's
log-binning, and of the scripts/dino_vlad.py calling pattern over the shim.  Tolerance 1e-4 relative."""
import numpy as np
import pytest
import torch
from torch.nn import functional as F

from oracle import anyloc_oracle as ao
from oracle import dino_v1_restated as d1
from tests import dino_v1_cases as cases
from tests.util import load_cases, matches_digest, rel_inf

pytestmark = pytest.mark.gpu
TOL = 1e-4
ENGINES = [("simt", "tf32x3"), ("simt", "f16x3"), ("auto", "tf32x3"), ("auto", "f16x3")]


@pytest.fixture(scope="module")
def dv(cuda):
    from anyloc_b200 import dino_v1
    return dino_v1


def _digest(g, key):
    return {k: g[f"{key}_{k}"] for k in ("shape", "sums", "pos", "vals")}


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("tag", list(cases.CASES))
def test_golden(dv, engine, tag):
    engine, precision = engine
    g = load_cases("dino_v1.npz")[tag]
    name, stride, H, W, B = cases.CASES[tag]
    ext = dv.ViTExtractor(name, stride, model=cases.model_for(name), device="cuda", gemm_engine=engine,
                          precision=precision)
    img = cases.image_for(tag).cuda()
    for layer in cases.LAYERS:
        for facet in cases.FACETS:
            out = ext.extract_descriptors(img, layer, facet)
            assert out.is_cuda
            assert matches_digest(out.cpu().numpy(), _digest(g, f"L{layer}_{facet}"), TOL), (layer, facet)
    assert tuple(ext.num_patches) == tuple(g["num_patches"]) and tuple(ext.load_size) == tuple(g["load_size"])
    out = ext.extract_descriptors(img, 11, "value", include_cls=True)
    assert matches_digest(out.cpu().numpy(), _digest(g, "L11_value_cls"), TOL)
    for facet in ("token", "key"):
        out = ext.extract_descriptors(img, 11, facet, bin=True)
        assert matches_digest(out.cpu().numpy(), _digest(g, f"L11_{facet}_bin"), TOL), facet


@pytest.mark.parametrize("precision", ["tf32x3", "f16x3"])
@pytest.mark.parametrize("name", list(d1.ARCHS))
def test_vs_oracle_strides(dv, precision, name):
    """every model at strides p, p/2, p/4 on a non-square image whose sides are multiples of nothing"""
    p = d1.ARCHS[name][3]
    model = d1.perturb(d1.build(name, seed=0, depth_override=3), seed=2)
    H, W = 5 * p + 3, 6 * p + 5
    img = torch.randn(2, 3, H, W, generator=torch.Generator().manual_seed(7))
    for stride in (p, p // 2, p // 4):
        ext = dv.ViTExtractor(name, stride, model=model, device="cuda", precision=precision)
        for facet in ("key", "token"):
            ref = d1.extract_descriptors(model, img, stride, 2, facet)
            err = rel_inf(ext.extract_descriptors(img.cuda(), 2, facet).cpu(), ref)
            assert err < TOL, (stride, facet, err)


@pytest.mark.parametrize("precision", ["tf32x3", "f16x3"])
def test_full_size_d1(dv, precision):
    """The d1 configuration (dino_vits8, stride 4, 224 x 298: a 55 x 73 grid, T = 4016 tokens, 32 key blocks with 48
    valid keys in the last) at full depth, layer 11, key and token; then dino_vitb8 at the same size, value."""
    img = torch.randn(1, 3, 224, 298, generator=torch.Generator().manual_seed(11))
    for name, facets in (("dino_vits8", ("key", "token")), ("dino_vitb8", ("value",))):
        model = d1.build(name, seed=0)
        ext = dv.ViTExtractor(name, 4, model=model, device="cuda", precision=precision)
        for facet in facets:
            out = ext.extract_descriptors(img.cuda(), 11, facet).cpu()
            assert out.shape == (1, 1, 55 * 73, model.embed_dim)
            ref = d1.extract_descriptors(model, img, 4, 11, facet)
            err = rel_inf(out, ref)
            print(f"d1 {name} {facet} {precision}: rel err {err:.2e}")
            assert err < TOL, (name, facet, err)
        del ext
        torch.cuda.empty_cache()


@pytest.mark.parametrize("gh,gw,C,B", [(1, 1, 8, 2), (1, 5, 8, 2), (2, 2, 8, 2), (3, 3, 8, 2), (5, 7, 8, 2),
                                       (7, 1, 12, 1), (9, 17, 36, 3), (16, 8, 64, 1), (55, 73, 384, 2)])
def test_log_bin_vs_oracle(dv, gh, gw, C, B):
    x = torch.randn(B, gh * gw, C, generator=torch.Generator().manual_seed(gh * 1000 + gw * 10 + C))
    out = dv.log_bin(x.cuda(), gh, gw)
    err = rel_inf(out.cpu(), d1.log_bin(x, gh, gw))
    assert err <= 1e-6, err


def test_log_bin_errors(dv):
    from anyloc_b200 import _lib
    x = torch.randn(1, 6, 8, device="cuda")
    with pytest.raises(_lib.AnylocError, match="hierarchy 3"):
        dv.log_bin(x, 2, 3, hierarchy=3)
    with pytest.raises(ValueError):
        dv.log_bin(torch.randn(1, 6, 6, device="cuda"), 2, 3)


def _dino_vlad_descs(extract, imgs, res, layer, facet, bin):
    """scripts/dino_vlad.py:171-182: per image interpolate, extract_descriptors, .squeeze().cpu(), then stack"""
    full = []
    for img in imgs:
        img = F.interpolate(img[None], res)
        full.append(extract(img, layer, facet, bin).squeeze().cpu())
    return torch.stack(full)


@pytest.mark.parametrize("K,bin", [(8, False), (4, True)])
def test_dino_vlad_pattern(dv, K, bin):
    from anyloc_b200 import utilities as u
    name, stride, layer, facet, res = "dino_vits8", 4, 2, "key", (48, 64)
    model = d1.perturb(d1.build(name, seed=0, depth_override=3), seed=3)
    imgs = torch.randn(4, 3, 96, 120, generator=torch.Generator().manual_seed(5))
    ext = dv.ViTExtractor(name, stride, model=model, device="cuda")
    ours = _dino_vlad_descs(lambda i, l, f, b: ext.extract_descriptors(i.cuda(), layer=l, facet=f, bin=b), imgs,
                            res, layer, facet, bin)
    ref = _dino_vlad_descs(lambda i, l, f, b: d1.extract_descriptors(model, i, stride, l, f, bin=b), imgs, res,
                           layer, facet, bin)
    assert ours.shape == ref.shape == (4, 11 * 15, 384 * (17 if bin else 1))
    assert rel_inf(ours, ref) < TOL
    np.random.seed(0)
    vlad = u.VLAD(K)
    vlad.fit(ours.reshape(-1, ours.shape[-1]))
    centers = vlad.c_centers.cpu()
    vl = vlad.generate_multi(ours)
    lab = torch.stack([vlad.kmeans.predict(f) for f in ours]).cpu()
    for b in range(ours.shape[0]):
        gap, lab64 = ao.label_margins(ref[b], centers)
        safe = gap > 1e-4
        assert torch.equal(lab[b][safe], lab64[safe])
    expect = torch.stack([ao.vlad_generate(f, centers, labels=l) for f, l in zip(ref, lab)])
    assert rel_inf(vl.cpu(), expect) < 5e-4       # features differ by ~1e-5; residual sums amplify


def test_dinov2_stride_zero_equals_stride_patch(cuda):
    from anyloc_b200 import vit
    from oracle import dinov2_restated as dr
    sd = dr.perturb(dr.build("dinov2_vits14", seed=0, depth_override=3), seed=1).state_dict()
    img = torch.randn(2, 3, 112, 154, generator=torch.Generator().manual_seed(2)).cuda()
    for pair in ("tf32", "f16"):
        a = vit.VitWeights("dinov2_vits14", sd, cuda, pair=pair)
        b = vit.VitWeights("dinov2_vits14", sd, cuda, pair=pair, stride=14)
        for facet in ("value", "token"):
            assert torch.equal(a.extract(img, 2, facet), b.extract(img, 2, facet)), (pair, facet)
