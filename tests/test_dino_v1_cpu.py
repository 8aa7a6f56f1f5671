"""CPU tests of the DINOv1 ViTExtractor path: the restated upstream model against transformers' independent ViT,
the oracle against the reference's own outputs (tests/golden/dino_v1.npz), and the product shim's host logic
(signature, attributes, layouts, errors) over a CPU double of the device forward."""
import contextlib
import inspect
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import dino_v1_restated as d1
from tests import dino_v1_cases as cases
from tests.util import ROOT, load_cases, matches_digest, rel_inf

TOL = 1e-5      # fp32 CPU arithmetic differs in the last bits between CPU types


@pytest.fixture(scope="module")
def golden():
    return load_cases("dino_v1.npz")


def _digest(g, key):
    return {k: g[f"{key}_{k}"] for k in ("shape", "sums", "pos", "vals")}


def test_restated_matches_transformers_vit():
    """stride = patch on a square 224 x 224 input: no resampling of the positional table on either side"""
    from transformers import ViTConfig, ViTModel
    depth = 2
    model = d1.perturb(d1.build("dino_vits16", seed=0, depth_override=depth), seed=1)
    cfg = ViTConfig(hidden_size=384, num_hidden_layers=depth, num_attention_heads=6, intermediate_size=1536,
                    hidden_act="gelu", layer_norm_eps=1e-6, image_size=224, patch_size=16, qkv_bias=True,
                    hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    hf = ViTModel(cfg, add_pooling_layer=False).eval()
    sd = model.state_dict()
    m = {"embeddings.cls_token": sd["cls_token"], "embeddings.position_embeddings": sd["pos_embed"],
         "embeddings.patch_embeddings.projection.weight": sd["patch_embed.proj.weight"],
         "embeddings.patch_embeddings.projection.bias": sd["patch_embed.proj.bias"],
         "layernorm.weight": sd["norm.weight"], "layernorm.bias": sd["norm.bias"]}
    for i in range(depth):
        p, q = f"blocks.{i}.", f"encoder.layer.{i}."
        w, b = sd[p + "attn.qkv.weight"].chunk(3), sd[p + "attn.qkv.bias"].chunk(3)
        for j, n in enumerate(("query", "key", "value")):
            m[q + f"attention.attention.{n}.weight"], m[q + f"attention.attention.{n}.bias"] = w[j], b[j]
        for src, dst in (("attn.proj", "attention.output.dense"), ("norm1", "layernorm_before"),
                         ("norm2", "layernorm_after"), ("mlp.fc1", "intermediate.dense"), ("mlp.fc2", "output.dense")):
            m[q + dst + ".weight"], m[q + dst + ".bias"] = sd[p + src + ".weight"], sd[p + src + ".bias"]
    hf.load_state_dict(m)
    img = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        ours = model.norm(model.blocks[1](model.blocks[0](model.prepare_tokens(img))))
        theirs = hf(pixel_values=img).last_hidden_state
        assert rel_inf(model(img), theirs[:, 0]) <= TOL
    assert rel_inf(ours, theirs) <= TOL


@pytest.mark.parametrize("tag", list(cases.CASES))
def test_oracle_matches_reference_golden(golden, tag):
    g = golden[tag]
    name, stride, H, W, B = cases.CASES[tag]
    model, img = cases.model_for(name), cases.image_for(tag)
    assert tuple(g["num_patches"]) == (1 + (H - model.patch_embed.patch_size) // stride,
                                       1 + (W - model.patch_embed.patch_size) // stride)
    for layer in cases.LAYERS:
        for facet in cases.FACETS:
            out = d1.extract_descriptors(model, img, stride, layer, facet).numpy()
            assert matches_digest(out, _digest(g, f"L{layer}_{facet}"), TOL), (layer, facet)
    out = d1.extract_descriptors(model, img, stride, 11, "value", include_cls=True).numpy()
    assert matches_digest(out, _digest(g, "L11_value_cls"), TOL)
    for facet in ("token", "key"):
        out = d1.extract_descriptors(model, img, stride, 11, facet, bin=True).numpy()
        assert matches_digest(out, _digest(g, f"L11_{facet}_bin"), TOL), facet


@pytest.mark.parametrize("gh,gw", cases.LOG_BIN_GRIDS)
def test_oracle_log_bin_matches_reference(golden, gh, gw):
    out = d1.log_bin(cases.log_bin_input(gh, gw), gh, gw)
    assert rel_inf(out, golden[f"logbin_{gh}x{gw}"]["out"]) <= 1e-6


def test_pos_embed_rule_matches_oracle():
    """vit.interpolate_pos_embed with DINOv1's pass-through rule (square pixels, not a square grid)"""
    from anyloc_b200 import vit
    model = cases.model_for("dino_vits16")
    for gh, gw, H, W in [(14, 14, 120, 120), (14, 14, 224, 230), (3, 4, 48, 64), (55, 73, 224, 298)]:
        ref = d1.pos_encoding(model, gh, gw, H, W)[0]
        assert torch.equal(vit.interpolate_pos_embed(model.pos_embed, gh, gw, H == W), ref), (gh, gw, H, W)


def test_random_state_dict_loads_into_restated_model():
    from anyloc_b200 import vit
    for name in ("dino_vits8", "dino_vitb16"):
        sd = vit.random_state_dict(name, seed=0, depth=2)
        assert not any("ls1" in k or "ls2" in k for k in sd)
        model = d1.VisionTransformer(name, depth_override=2)
        model.load_state_dict(sd, strict=True)
        assert float(sd["cls_token"].std()) > 1e-3          # trunc_normal .02, not DINOv2's N(0, 1e-6)


class _DoubleVit:
    """stands in for vit.VitWeights: the restated model with the given state_dict, run by the oracle"""

    def __init__(self, name, state_dict, device, depth=None, pair="tf32", stride=None):
        self.model, self.stride = d1.from_state_dict(state_dict, name), stride
        self.depth = len(self.model.blocks)

    def extract(self, img, layer, facet="value", use_cls=False, norm_descs=True, engine="auto", desc=None):
        with torch.no_grad():
            x, _ = d1.facet_tokens(self.model, img.float(), self.stride, layer, facet)
        if desc == "interleaved" and facet != "token":
            x = d1.interleave_heads(x, self.model.blocks[0].attn.num_heads)
        return x if use_cls else x[:, 1:]


@contextlib.contextmanager
def _cpu_double():
    from anyloc_b200 import _lib, dino_v1, vit
    saved = [(_lib, "require_cuda", _lib.require_cuda), (vit, "VitWeights", vit.VitWeights),
             (dino_v1, "log_bin", dino_v1.log_bin)]
    _lib.require_cuda = lambda device=None: torch.device("cpu")
    vit.VitWeights = _DoubleVit
    dino_v1.log_bin = lambda x, gh, gw, hierarchy=2: d1.log_bin(x, gh, gw)
    try:
        yield dino_v1
    finally:
        for obj, name, old in saved:
            setattr(obj, name, old)


def test_shim_signature_and_attributes(golden):
    from anyloc_b200.dino_v1 import ViTExtractor
    sig = inspect.signature(ViTExtractor.__init__)
    params = list(sig.parameters.values())[1:]
    assert [p.name for p in params[:4]] == ["model_type", "stride", "model", "device"]    # dino_extractor.py:42
    assert [p.default for p in params[:4]] == ["dino_vits8", 4, None, "cuda"]
    assert all(p.kind is p.KEYWORD_ONLY for p in params[4:])
    assert {p.name for p in params[4:]} == {"weights", "gemm_engine", "precision"}
    for m in ("preprocess", "extract_descriptors", "_extract_features", "_log_bin", "extract_saliency_maps"):
        assert callable(getattr(ViTExtractor, m))
    tag = "vits8_s4_60x76"
    name, stride, H, W, B = cases.CASES[tag]
    g = golden[tag]
    with _cpu_double() as dv:
        ext = dv.ViTExtractor(name, stride, model=cases.model_for(name), device="cpu")
        assert (ext.p, ext.stride, ext.model_type, ext.device) == (8, (4, 4), name, "cpu")
        assert ext.mean == (0.485, 0.456, 0.406) and ext.std == (0.229, 0.224, 0.225)
        assert ext.load_size is None and ext.num_patches is None
        img = cases.image_for(tag)
        out = ext.extract_descriptors(img, 11, "key")
        assert matches_digest(out.numpy(), _digest(g, "L11_key"), TOL)
        assert ext.load_size == (H, W) and tuple(ext.num_patches) == tuple(g["num_patches"])
        assert matches_digest(ext.extract_descriptors(img, 11, "key", bin=True).numpy(), _digest(g, "L11_key_bin"), TOL)
        assert matches_digest(ext.extract_descriptors(img, 11, "value", include_cls=True).numpy(),
                              _digest(g, "L11_value_cls"), TOL)
        feats = ext._extract_features(img, [11], "key")
        assert len(feats) == 1 and feats[0].shape == (B, 6, 1 + 14 * 18, 64)
        # extract_descriptors = the reference's permute/flatten of the hook output (dino_extractor.py:329)
        ref = feats[0][:, :, 1:].permute(0, 2, 3, 1).flatten(-2).unsqueeze(1)
        assert torch.equal(ref, out)
        assert torch.equal(ext._log_bin(feats[0][:, :, 1:]), ext.extract_descriptors(img, 11, "key", bin=True))
        assert ext._extract_features(img, [5], "token")[0].shape == (B, 1 + 14 * 18, 384)
        timm = dv.ViTExtractor("vit_small_patch8_224", 8, model=cases.model_for(name), device="cpu")
        assert timm.mean == (0.5, 0.5, 0.5) and timm.stride == (8, 8)
        # preprocess: LANCZOS resize of the shorter side, ToTensor, Normalize
        u8 = (np.random.default_rng(0).random((30, 40, 3)) * 255).astype(np.uint8)
        x, pil = ext.preprocess(u8, 24)
        assert x.shape == (1, 3, 24, 32) and pil.size == (32, 24)
        x, _ = ext.preprocess(u8)
        ref = (torch.from_numpy(u8).permute(2, 0, 1).float() / 255 - torch.tensor(ext.mean)[:, None, None]) / \
            torch.tensor(ext.std)[:, None, None]
        assert torch.allclose(x[0], ref, atol=1e-6)


def test_shim_errors():
    from anyloc_b200 import _lib
    from anyloc_b200.dino_v1 import ViTExtractor
    with pytest.raises(_lib.AnylocError):
        ViTExtractor("dino_vits8", 4, device="cpu")                       # CUDA only, loud
    with pytest.raises(AssertionError):
        ViTExtractor("dino_vits8", 3)                                     # stride must divide the patch
    with pytest.raises(ValueError):
        ViTExtractor("dino_vitl8", 4)                                     # unknown model
    with _cpu_double() as dv:
        ext = dv.ViTExtractor("dino_vits16", 8, model=cases.model_for("dino_vits16"), device="cpu")
        img = cases.image_for("vits16_s8_120x120")
        with pytest.raises(AssertionError):
            ext.extract_descriptors(img, 11, "key", bin=True, include_cls=True)
        with pytest.raises(AssertionError):
            ext.extract_descriptors(img, 11, "attn")
        with pytest.raises(_lib.AnylocError, match="out of scope"):
            ext._extract_features(img, [11], "attn")
        with pytest.raises(_lib.AnylocError, match="out of scope"):
            ext.extract_saliency_maps(img)


def test_dropin_resolves_dino_extractor():
    code = ("import sys; sys.path.insert(0, %r); from dino_extractor import ViTExtractor; "
            "print(ViTExtractor.__module__)" % os.path.join(ROOT, "anyloc_b200", "dropin"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd="/tmp")
    assert out.returncode == 0, out.stderr
    assert out.stdout.strip().splitlines()[-1] == "anyloc_b200.dino_v1"
