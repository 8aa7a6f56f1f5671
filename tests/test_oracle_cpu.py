"""CPU tests: the oracle restatement against the committed golden vectors (generated from the
reference's own code, tests/golden/make_golden.py) and the restated ViT against the independent HuggingFace port."""
import numpy as np
import pytest
import torch

from oracle import anyloc_oracle as ao
from oracle import dinov2_restated as dr
from oracle import fpk_restated as fpk
from tests.util import (PCA_CHECK_KWARGS, case_kwargs, load_cases, pca_check_inputs, rel_inf,
                        vlad_topk_check_inputs)

# Goldens that went through fp32 matrix products or LAPACK were made on one CPU; another CPU's kernels round
# differently in the last bits (about 1e-6 relative here).
CPU_TOL = 1e-5


@pytest.mark.parametrize("name", sorted(n for n in load_cases("vlad.npz") if not n.startswith("multi")))
def test_vlad_oracle_matches_golden(name):
    c = load_cases("vlad.npz")[name]
    kw = case_kwargs(c)
    out = ao.vlad_generate(torch.from_numpy(c["x"]), torch.from_numpy(c["centers"]), **kw)
    lab = ao.vlad_labels(torch.from_numpy(c["x"]), torch.from_numpy(c["centers"]), kw.get("dist_mode", "cosine"))
    assert torch.equal(lab, torch.from_numpy(c["labels"]))
    assert torch.equal(out, torch.from_numpy(c["out"]))          # same ops, same order: bit-exact


def test_vlad_multi_oracle_matches_golden():
    c = load_cases("vlad.npz")["multi_b4_n50_d32_k6"]
    out = ao.vlad_generate_multi(torch.from_numpy(c["x"]), torch.from_numpy(c["centers"]))
    assert torch.equal(out, torch.from_numpy(c["out"]))


@pytest.mark.parametrize("name", sorted(load_cases("vlad_soft.npz")))
def test_vlad_soft_oracle_matches_golden(name):
    """Soft branch (utilities.py:862-887): restatement bit-exact with the reference's output; the closed form the
    CUDA path uses, V_k = K sum_q a_qk x^_q - (sum_q a_qk) sum_c c_c, agrees in fp64."""
    c = load_cases("vlad_soft.npz")[name]
    kw = case_kwargs(c)
    xs, ce = torch.from_numpy(c["x"]), torch.from_numpy(c["centers"])
    ref = torch.from_numpy(c["out"])
    if xs.dim() == 2:
        xs, ref = xs[None], ref[None]
    for x, r in zip(xs, ref):
        assert torch.equal(ao.vlad_generate_soft(x, ce, **kw), r)
        v = ao.vlad_generate_soft_closed(x, ce, **kw)
        assert float((v - r.double()).abs().max() / r.abs().max()) < 1e-5


@pytest.mark.parametrize("name", sorted(load_cases("preprocess.npz")))
def test_preprocess_oracle_matches_golden(name):
    """ToTensor + Normalize + CenterCrop restated; golden outputs come from torchvision itself."""
    c = load_cases("preprocess.npz")[name]
    out = ao.preprocess(torch.from_numpy(c["img"]))
    assert out.shape == c["out"].shape
    assert torch.equal(out, torch.from_numpy(c["out"]))


def test_vlad_golden_properties():
    c = load_cases("vlad.npz")["emptyclusters_n10_d32_k16"]
    out = torch.from_numpy(c["out"]).reshape(16, 32)
    used = sorted(set(c["labels"].tolist()))
    for k in range(16):
        if k in used:
            assert abs(float(out[k].norm()) - 1 / len(used) ** 0.5) < 1e-6
        else:
            assert float(out[k].abs().max()) == 0.0          # utilities.py:840,854-855
    t = load_cases("vlad.npz")["ties_zero_n40_d32_k4"]
    assert 2 not in set(t["labels"].tolist())                # duplicate centre: lowest index wins
    assert t["labels"][3] == 0 and t["labels"][7] == 0       # all-zero descriptor -> label 0


def test_topk_oracle_matches_golden():
    g = load_cases("topk.npz")
    db, qu = torch.from_numpy(g[""]["db"]), torch.from_numpy(g[""]["qu"])
    gt = np.empty(len(g[""]["gt"]), dtype=object)
    for i, row in enumerate(g[""]["gt"]):
        gt[i] = row
    for method in ("cosine", "l2"):
        d, i, r = ao.get_top_k_recall([1, 3, 5], db, qu, gt, method=method)
        assert torch.equal(i, torch.from_numpy(g[method]["idx"]))
        assert torch.equal(d, torch.from_numpy(g[method]["dist"]))
        assert np.allclose([r[k] for k in (1, 3, 5)], g[method]["recalls"])
    # duplicate DB rows 4 and 11: lowest index first
    idx = g["cosine"]["idx"]
    for row in idx:
        row = row.tolist()
        if 4 in row and 11 in row:
            assert row.index(4) < row.index(11)
    d, i, r = ao.get_top_k_recall([2], db, qu[0], gt, norm_descs=False, use_percentage=False)
    assert torch.equal(i, torch.from_numpy(g["single"]["idx"]))
    assert r[2] == g["single"]["recalls"][0]


def test_fit_restated_matches_golden():
    g = load_cases("fit.npz")[""]
    x = torch.nn.functional.normalize(torch.from_numpy(g["x"]))
    np.random.seed(42)
    km = fpk.KMeans(5, mode="cosine")
    km.fit(x)
    assert torch.allclose(km.centroids, torch.from_numpy(g["centers"]), atol=0, rtol=0)


@pytest.mark.parametrize("tag,name,depth,layer", [("vits14_l9_56x70", "dinov2_vits14", None, 9),
                                                   ("vitg14_d2_l1_42x42", "dinov2_vitg14", 2, 1)])
def test_extract_oracle_matches_golden(tag, name, depth, layer):
    g = load_cases("extract.npz")[tag]
    model = dr.perturb(dr.build(name, seed=0, depth_override=depth), seed=1)
    img = torch.from_numpy(g["img"])
    for facet in ("value", "key", "query", "token"):
        out = ao.extract_features(model, img, layer, facet)
        # early exit == full forward + hook (SURVEY.md 8c): identical ops on the path that matters, bit for bit
        assert torch.equal(out, ao.extract_features_full_forward(model, img, layer, facet)), facet
        assert rel_inf(out, g[facet]) < CPU_TOL, facet
    out = ao.extract_features(model, img, layer, "value", use_cls=True, norm_descs=False)
    assert torch.equal(out, ao.extract_features_full_forward(model, img, layer, "value", use_cls=True, norm_descs=False))
    assert rel_inf(out, g["value_cls_nonorm"]) < CPU_TOL


def test_oracle_matches_verbatim_reference():
    """oracle VLAD.generate and get_top_k_recall == the reference's own (tests/golden/reference_checks.npz), bit for bit"""
    g = load_cases("reference_checks.npz")
    vlads, db, qu, gt = vlad_topk_check_inputs()
    for j, (x, c) in enumerate(vlads):
        assert torch.equal(torch.from_numpy(g[f"vlad{j}"]["out"]), ao.vlad_generate(x, c))
    d2, i2, r2 = ao.get_top_k_recall([1, 4], db, qu, gt)
    assert torch.equal(torch.from_numpy(g["topk"]["idx"]), i2) and torch.equal(torch.from_numpy(g["topk"]["dist"]), d2)
    assert r2 == dict(zip([1, 4], g["topk"]["recalls"].tolist()))


def _hf_model_from(model, name, H, W, depth):
    from transformers import Dinov2Config, Dinov2Model
    dim, _, heads, ffn = dr.ARCHS[name]
    cfg = Dinov2Config(hidden_size=dim, num_hidden_layers=depth, num_attention_heads=heads, mlp_ratio=4,
                       image_size=H, patch_size=14, use_swiglu_ffn=(ffn != "mlp"), layer_norm_eps=1e-6,
                       hidden_act="gelu", qkv_bias=True, layerscale_value=1.0,
                       attn_implementation="eager")
    hf = Dinov2Model(cfg).eval()
    sd = {k: v for k, v in model.state_dict().items()}
    with torch.no_grad():
        e = hf.embeddings
        e.cls_token.copy_(sd["cls_token"])
        x = torch.zeros(1, 1 + (H // 14) * (W // 14), dim)
        e.position_embeddings.copy_(model.interpolate_pos_encoding(x, H, W))
        e.patch_embeddings.projection.weight.copy_(sd["patch_embed.proj.weight"])
        e.patch_embeddings.projection.bias.copy_(sd["patch_embed.proj.bias"])
        for i, layer in enumerate(hf.encoder.layer):
            p = f"blocks.{i}."
            layer.norm1.weight.copy_(sd[p + "norm1.weight"]); layer.norm1.bias.copy_(sd[p + "norm1.bias"])
            layer.norm2.weight.copy_(sd[p + "norm2.weight"]); layer.norm2.bias.copy_(sd[p + "norm2.bias"])
            w, b = sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"]
            att = layer.attention.attention
            for j, lin in enumerate((att.query, att.key, att.value)):
                lin.weight.copy_(w[j * dim:(j + 1) * dim]); lin.bias.copy_(b[j * dim:(j + 1) * dim])
            layer.attention.output.dense.weight.copy_(sd[p + "attn.proj.weight"])
            layer.attention.output.dense.bias.copy_(sd[p + "attn.proj.bias"])
            layer.layer_scale1.lambda1.copy_(sd[p + "ls1.gamma"])
            layer.layer_scale2.lambda1.copy_(sd[p + "ls2.gamma"])
            if ffn == "mlp":
                layer.mlp.fc1.weight.copy_(sd[p + "mlp.fc1.weight"]); layer.mlp.fc1.bias.copy_(sd[p + "mlp.fc1.bias"])
                layer.mlp.fc2.weight.copy_(sd[p + "mlp.fc2.weight"]); layer.mlp.fc2.bias.copy_(sd[p + "mlp.fc2.bias"])
            else:
                layer.mlp.weights_in.weight.copy_(sd[p + "mlp.w12.weight"]); layer.mlp.weights_in.bias.copy_(sd[p + "mlp.w12.bias"])
                layer.mlp.weights_out.weight.copy_(sd[p + "mlp.w3.weight"]); layer.mlp.weights_out.bias.copy_(sd[p + "mlp.w3.bias"])
    return hf


@pytest.mark.parametrize("name,depth", [("dinov2_vits14", 3), ("dinov2_vitg14", 2)])
def test_restated_vit_matches_hf_port(name, depth):
    """Independent pin of the block arithmetic: HuggingFace's Dinov2Model with remapped weights."""
    H = W = 56
    model = dr.perturb(dr.build(name, seed=0, depth_override=depth), seed=1)
    hf = _hf_model_from(model, name, H, W, depth)
    img = torch.randn(2, 3, H, W, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        hs = hf(pixel_values=img, output_hidden_states=True).hidden_states   # [emb, blk0, blk1, ...]
    tok = ao.extract_features(model, img, depth - 1, "token", use_cls=True, norm_descs=False)
    assert torch.allclose(tok, hs[depth], atol=2e-5, rtol=1e-5)


def test_reduce_pca_matches_reference():
    """oracle.reduce_pca == the reference's reduce_pca (utilities.py:522-586), both branches
    (tests/golden/reference_checks.npz; bit for bit on the CPU that made it)."""
    g = load_cases("reference_checks.npz")
    tr, te = pca_check_inputs()
    for j, kw in enumerate(PCA_CHECK_KWARGS):
        b = ao.reduce_pca(tr.copy(), te.copy(), 8, **kw)
        assert rel_inf(b[0], g[f"pca{j}"]["train"]) < CPU_TOL and rel_inf(b[1], g[f"pca{j}"]["test"]) < CPU_TOL


def test_preprocess_resize_matches_torchvision_golden():
    """oracle.preprocess(resize=...) == torchvision's ToTensor + Normalize + antialiased tensor resize + CenterCrop
    (tests/golden/preprocess_resize.npz, made by torchvision itself), bit for bit."""
    for name, c in load_cases("preprocess_resize.npz").items():
        out = ao.preprocess(c["img"], resize=tuple(int(v) for v in c["size"]), interpolation=name.split("_")[0])
        assert torch.equal(out, torch.from_numpy(c["out"])), name


def test_oracle_reproduces_reference_driver_run():
    """tests/golden/build_vlads.npz holds what the reference's UNMODIFIED build_vlads (scripts/dino_v2_vlad.py:124-303)
    produced over its own utilities.py; the oracle restatements (extractor, fpk k-means, VLAD, top-k) driven the same way
    must reproduce it -- this is what the GPU parity tests are then measured against."""
    from tests import dropin_harness as H
    ds = H.SyntheticVprDataset()
    model = dr.perturb(dr.build("dinov2_vits14", seed=0, depth_override=3), seed=3)
    imgs = torch.stack([ds[i][0][:, 2:58, 2:72] for i in range(len(ds))])        # T.CenterCrop((56, 70)) of 60 x 75
    feats = ao.extract_features(model, imgs, 2, "value")
    for tag, g in load_cases("build_vlads.npz").items():
        np.random.seed(42)
        km = fpk.KMeans(4, mode="cosine")
        km.fit(torch.nn.functional.normalize(feats[:ds.database_num].reshape(-1, 384), dim=1))
        assert torch.allclose(km.centroids, torch.from_numpy(g["c_centers"]), atol=1e-6)
        gen = ao.vlad_generate if tag == "hard" else ao.vlad_generate_soft
        vl = torch.stack([gen(f, km.centroids) for f in feats])
        assert torch.allclose(vl[:ds.database_num], torch.from_numpy(g["db_vlads"]), atol=2e-6)
        assert torch.allclose(vl[ds.database_num:], torch.from_numpy(g["qu_vlads"]), atol=2e-6)
        d, i = ao.top_k(vl[:ds.database_num], vl[ds.database_num:], 3)
        assert np.array_equal(i.numpy(), g["idx"])
