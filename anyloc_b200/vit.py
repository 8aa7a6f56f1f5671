"""Host side of the ViT extractors: weight preparation (tf32 hi/lo split, SwiGLU row
interleave, patch-embed flattening), positional-embedding interpolation (upstream
`interpolate_pos_encoding`, done once per resolution) and the call into
`anyloc_vit_extract` (include/anyloc_b200.h).

Reference: /root/reference/utilities.py:219-288 (DinoV2ExtractFeatures) and the hub model it
loads (facebookresearch/dinov2; spec in SURVEY.md Appendix A); /root/reference/dino_extractor.py
(ViTExtractor) and the DINOv1 models it loads (facebookresearch/dino, or timm weights in them).
DINOv1 blocks are the DINOv2 MLP blocks without LayerScale (uploaded as ones: 1.0f*y == y).
"""
import ctypes as C
import math
import os

import torch
from torch.nn import functional as F

from . import _lib

class Arch(tuple):
    """(embed_dim, depth, heads, ffn kind) -- what unpacking an ARCHS entry yields -- plus the patch size, the side
    of the pretrained positional-embedding grid and the family ("dinov2" or "dino", i.e. DINOv1)."""

    def __new__(cls, dim, depth, heads, kind, patch, pos_grid, family):
        self = super().__new__(cls, (dim, depth, heads, kind))
        self.patch, self.pos_grid, self.family = patch, pos_grid, family
        return self


ARCHS = {
    "dinov2_vits14": Arch(384, 12, 6, "mlp", 14, 37, "dinov2"),        # pretrained at 518x518
    "dinov2_vitb14": Arch(768, 12, 12, "mlp", 14, 37, "dinov2"),
    "dinov2_vitl14": Arch(1024, 24, 16, "mlp", 14, 37, "dinov2"),
    "dinov2_vitg14": Arch(1536, 40, 24, "swiglufused", 14, 37, "dinov2"),
    "dino_vits8": Arch(384, 12, 6, "mlp", 8, 28, "dino"),               # pretrained at 224x224
    "dino_vits16": Arch(384, 12, 6, "mlp", 16, 14, "dino"),
    "dino_vitb8": Arch(768, 12, 12, "mlp", 8, 28, "dino"),
    "dino_vitb16": Arch(768, 12, 12, "mlp", 16, 14, "dino"),
}
# timm checkpoints ViTExtractor loads into the DINOv1 architecture of the same shape (dino_extractor.py:88-99)
TIMM_ARCH = {"vit_small_patch16_224": "dino_vits16", "vit_small_patch8_224": "dino_vits8",
             "vit_base_patch16_224": "dino_vitb16", "vit_base_patch8_224": "dino_vitb8"}
PATCH = 14              # DINOv2
POS_GRID = 37
INTERP_OFFSET = 0.1     # upstream interpolate_offset (DINOv1 adds the same 0.1)


def ffn_hidden(dim, kind):
    return 4 * dim if kind == "mlp" else (int(4 * dim * 2 / 3) + 7) // 8 * 8


def random_state_dict(name, seed=0, device="cpu", depth=None):
    """Random weights with the upstream init recipe (trunc_normal std .02 for Linear / pos_embed,
    cls ~ N(0,1e-6) for DINOv2 and trunc_normal .02 for DINOv1, zero bias, LayerNorm (1,0), LayerScale
    1.0 for DINOv2, none for DINOv1), generated directly on `device`.
    Synthetic-benchmark use only: no pretrained checkpoint can be fetched offline."""
    arch = ARCHS[name]
    dim, full_depth, heads, kind = arch
    v1 = arch.family == "dino"
    depth = full_depth if depth is None else depth
    hid = ffn_hidden(dim, kind)
    g = torch.Generator(device=device).manual_seed(seed)

    def tn(*shape):
        t = torch.empty(*shape, device=device, dtype=torch.float32)
        # trunc_normal_(std=.02, a=-2, b=2): the +-2 bounds are 100 sigma away -> plain normal
        return t.normal_(0.0, 0.02, generator=g)

    def zeros(*s):
        return torch.zeros(*s, device=device)

    def ones(*s):
        return torch.ones(*s, device=device)

    sd = {
        "cls_token": tn(1, 1, dim) if v1 else torch.empty(1, 1, dim, device=device).normal_(0.0, 1e-6, generator=g),
        "pos_embed": tn(1, 1 + arch.pos_grid ** 2, dim),
        "patch_embed.proj.weight": tn(dim, 3, arch.patch, arch.patch),
        "patch_embed.proj.bias": zeros(dim),
    }
    for i in range(depth):
        p = f"blocks.{i}."
        sd[p + "norm1.weight"], sd[p + "norm1.bias"] = ones(dim), zeros(dim)
        sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"] = tn(3 * dim, dim), zeros(3 * dim)
        sd[p + "attn.proj.weight"], sd[p + "attn.proj.bias"] = tn(dim, dim), zeros(dim)
        if not v1:
            sd[p + "ls1.gamma"] = ones(dim)
        sd[p + "norm2.weight"], sd[p + "norm2.bias"] = ones(dim), zeros(dim)
        if kind == "mlp":
            sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"] = tn(hid, dim), zeros(hid)
            sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"] = tn(dim, hid), zeros(dim)
        else:
            sd[p + "mlp.w12.weight"], sd[p + "mlp.w12.bias"] = tn(2 * hid, dim), zeros(2 * hid)
            sd[p + "mlp.w3.weight"], sd[p + "mlp.w3.bias"] = tn(dim, hid), zeros(dim)
        if not v1:
            sd[p + "ls2.gamma"] = ones(dim)
    if v1:
        sd["norm.weight"], sd["norm.bias"] = ones(dim), zeros(dim)
    return sd


def interpolate_pos_embed(pos_embed, gh, gw, square=None):
    """Upstream interpolate_pos_encoding for a gh x gw patch grid (gh rows, gw columns): DINOv2's
    DinoVisionTransformer and DINOv1's VisionTransformer (also as patched by dino_extractor.py:105-138,
    the same rule).  pos_embed [1, 1+m*m, D] -> [1+gh*gw, D].  The table passes through unchanged only
    when the grid has m*m cells AND the image is square in pixels (`square`; by default gh == gw, which
    is the same thing when H and W are multiples of the patch) -- a non-square image whose strided grid
    happens to have m*m cells is still resampled.  Otherwise bicubic with the given scale factors
    ((g+0.1)/m, align_corners=False) driving the coordinate map."""
    pos_embed = pos_embed.detach().float().cpu()
    n = pos_embed.shape[1] - 1
    m = int(math.sqrt(n))
    if gh * gw == n and (gh == gw if square is None else square):
        return pos_embed[0].contiguous()
    dim = pos_embed.shape[-1]
    cls_pos, patch_pos = pos_embed[:, 0], pos_embed[:, 1:]
    sy, sx = float(gh + INTERP_OFFSET) / m, float(gw + INTERP_OFFSET) / m
    patch_pos = F.interpolate(patch_pos.reshape(1, m, m, dim).permute(0, 3, 1, 2),
                              scale_factor=(sy, sx), mode="bicubic", antialias=False)
    if tuple(patch_pos.shape[-2:]) != (gh, gw):
        raise _lib.AnylocError(f"pos-embed interpolation produced {tuple(patch_pos.shape[-2:])}, wanted {(gh, gw)}")
    patch_pos = patch_pos.permute(0, 2, 3, 1).reshape(-1, dim)
    return torch.cat([cls_pos, patch_pos], dim=0).contiguous()


class VitWeights:
    """Device-resident, kernel-ready weights of one DINOv2 or DINOv1 backbone (blocks 0..depth-1).
    `stride` (DINOv1 only) is the patch-embedding stride; None keeps the non-overlapping DINOv2 contract
    (H, W multiples of the patch).  DINOv1 state dicts carry no LayerScale (ones are uploaded); their
    `norm.*` and `head.*` entries are not needed by any facet and are ignored."""

    def __init__(self, name, state_dict, device, depth=None, pair="tf32", stride=None):
        if name not in ARCHS:
            raise ValueError(f"unknown ViT model {name!r}; expected one of {sorted(ARCHS)}")
        if pair not in _lib.PAIR:
            raise ValueError(f"pair must be one of {sorted(_lib.PAIR)}, got {pair!r}")
        arch = ARCHS[name]
        self.patch, self.family = arch.patch, arch.family
        if stride is not None and (stride <= 0 or self.patch % stride):
            raise ValueError(f"stride {stride} must divide the patch size {self.patch}")
        self.stride = stride
        self.name = name
        self.pair = pair
        self.device = _lib.require_cuda(device)
        self.dim, full_depth, self.heads, self.ffn_kind = arch
        n_blocks = 1 + max([int(k.split(".")[1]) for k in state_dict if k.startswith("blocks.")], default=-1)
        self.depth = min(n_blocks, full_depth if depth is None else depth)
        self.hidden = ffn_hidden(self.dim, self.ffn_kind)
        self._keep = []          # owning references of every device tensor handed to the C side
        self._pos_cache = {}
        lib = _lib.load()
        self.patch_k = lib.anyloc_vit_patch_k(self.patch)
        dev = self.device

        def f32(t):
            return t.detach().to(device=dev, dtype=torch.float32).contiguous()

        def split(t):
            """-> (hi, lo, alpha): the kernel-ready pair of a weight matrix and the accumulator scale
            1/(s_act*s_w) its GEMM epilogue applies (1.0 for tf32 pairs)."""
            t = f32(t)
            with torch.cuda.device(dev):
                if pair == "tf32":
                    hi, lo = torch.empty_like(t), torch.empty_like(t)
                    _lib.check(lib.anyloc_split_tf32(_lib.ptr(t), _lib.ptr(hi), _lib.ptr(lo), t.numel(),
                                                     _lib.stream_ptr()), "split_tf32")
                    alpha = 1.0
                else:
                    # per-tensor power-of-two scale: largest |w| lands in [8192, 16384) -- far from fp16's 65504
                    # ceiling, and typical weights sit well inside the normal range (hi+lo keeps ~22 bits)
                    amax = float(t.abs().max().item())
                    s_w = 2.0 ** math.floor(math.log2(16384.0 / amax)) if amax > 0 else 1.0
                    hi = torch.empty(t.shape, dtype=torch.float16, device=dev)
                    lo = torch.empty(t.shape, dtype=torch.float16, device=dev)
                    _lib.check(lib.anyloc_split_f16(_lib.ptr(t), _lib.ptr(hi), _lib.ptr(lo), t.numel(),
                                                    C.c_float(s_w), _lib.stream_ptr()), "split_f16")
                    alpha = 1.0 / (_lib.ACT_SCALE * s_w)
            self._keep += [hi, lo]
            return hi, lo, alpha

        def keep(t):
            t = f32(t)
            self._keep.append(t)
            return t

        sd = state_dict
        pw = f32(sd["patch_embed.proj.weight"]).reshape(self.dim, -1)
        pw = F.pad(pw, (0, self.patch_k - pw.shape[1]))
        self.patch_w = split(pw)
        patch_alpha = self.patch_w[2]
        self.patch_b = keep(sd["patch_embed.proj.bias"])
        self.cls_token = keep(sd["cls_token"].reshape(-1))
        self.pos_embed = sd["pos_embed"].detach().float().cpu()
        self.blocks = (_lib.VitBlock * self.depth)()
        for i in range(self.depth):
            p = f"blocks.{i}."
            blk = self.blocks[i]

            def put(field, t):
                setattr(blk, field, t.data_ptr())

            put("ln1_w", keep(sd[p + "norm1.weight"])); put("ln1_b", keep(sd[p + "norm1.bias"]))
            hi, lo, blk.qkv_alpha = split(sd[p + "attn.qkv.weight"]); put("qkv_w_hi", hi); put("qkv_w_lo", lo)
            put("qkv_b", keep(sd[p + "attn.qkv.bias"]))
            hi, lo, blk.proj_alpha = split(sd[p + "attn.proj.weight"]); put("proj_w_hi", hi); put("proj_w_lo", lo)
            put("proj_b", keep(sd[p + "attn.proj.bias"]))
            no_ls = torch.ones(self.dim)
            put("ls1", keep(no_ls if self.family == "dino" else sd[p + "ls1.gamma"]))
            put("ln2_w", keep(sd[p + "norm2.weight"])); put("ln2_b", keep(sd[p + "norm2.bias"]))
            if self.ffn_kind == "mlp":
                w_in, b_in = sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"]
                w_out, b_out = sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"]
            else:
                # interleave so GEMM columns (2j, 2j+1) = (x1_j, x2_j): the SwiGLU epilogue needs
                # both halves of `w12(x).chunk(2)` for the same j in one thread
                h = self.hidden
                perm = torch.stack([torch.arange(h), torch.arange(h) + h], dim=1).reshape(-1)
                w_in = sd[p + "mlp.w12.weight"].detach().cpu()[perm]
                b_in = sd[p + "mlp.w12.bias"].detach().cpu()[perm]
                w_out, b_out = sd[p + "mlp.w3.weight"], sd[p + "mlp.w3.bias"]
            hi, lo, blk.in_alpha = split(w_in); put("in_w_hi", hi); put("in_w_lo", lo); put("in_b", keep(b_in))
            hi, lo, blk.out_alpha = split(w_out); put("out_w_hi", hi); put("out_w_lo", lo); put("out_b", keep(b_out))
            put("ls2", keep(no_ls if self.family == "dino" else sd[p + "ls2.gamma"]))
        self.cfg = _lib.VitCfg(self.dim, self.depth, self.heads, _lib.FFN[self.ffn_kind], self.hidden, self.patch,
                               _lib.PAIR[pair], stride or 0)
        self.struct = _lib.VitWeightsStruct(self.patch_w[0].data_ptr(), self.patch_w[1].data_ptr(),
                                            self.patch_b.data_ptr(), self.cls_token.data_ptr(), self.blocks,
                                            patch_alpha)
        torch.cuda.synchronize(dev)

    def grid(self, H, W):
        """patch grid (gh, gw) of an H x W image; raises ValueError where the embedding does not apply"""
        P = self.patch
        if self.stride is None:
            if H % P or W % P:
                raise ValueError(f"image size {(H, W)} is not a multiple of the patch size {P}")
            return H // P, W // P
        if H < P or W < P:
            raise ValueError(f"image size {(H, W)} is smaller than the patch size {P}")
        return 1 + (H - P) // self.stride, 1 + (W - P) // self.stride

    def pos_for(self, gh, gw, square=None):
        key = (gh, gw, square)
        if key not in self._pos_cache:
            self._pos_cache[key] = interpolate_pos_embed(self.pos_embed, gh, gw, square).to(self.device)
        return self._pos_cache[key]

    def extract(self, img, layer, facet="value", use_cls=False, norm_descs=True, engine="auto", desc=None):
        """img [B,3,H,W] fp32 on self.device -> [B, N(+1), D] fp32 (utilities.py:263-285).  `desc` ("plain", "l2"
        or "interleaved": ViTExtractor's head-interleaved q/k/v channel order, dino_extractor.py:329) overrides
        norm_descs."""
        if img.dim() != 4 or img.shape[1] != 3:
            raise ValueError(f"expected an image batch [B,3,H,W], got {tuple(img.shape)}")
        B, _, H, W = img.shape
        gh, gw = self.grid(H, W)
        if not 0 <= layer < self.depth:
            raise IndexError(f"layer {layer} out of range for {self.name} with {self.depth} blocks loaded")
        desc_mode = _lib.DESC[desc] if desc is not None else int(bool(norm_descs))
        img = img.to(device=self.device, dtype=torch.float32).contiguous()
        n_out = gh * gw + (1 if use_cls else 0)
        out = torch.empty(B, n_out, self.dim, device=self.device, dtype=torch.float32)
        lib = _lib.load()
        pos = self.pos_for(gh, gw, None if self.stride is None else H == W)
        with torch.cuda.device(self.device):
            nbytes = lib.anyloc_vit_workspace_bytes(C.byref(self.cfg), B, H, W)
            ws = _lib.workspaces.get(self.device, nbytes, "vit")
            rc = lib.anyloc_vit_extract(C.byref(self.cfg), C.byref(self.struct), _lib.ptr(img), B, H, W,
                                        _lib.ptr(pos), layer, _lib.FACET[facet], int(bool(use_cls)),
                                        desc_mode, _lib.ptr(out), _lib.ptr(ws), ws.numel(),
                                        _lib.ENGINE[engine], _lib.stream_ptr())
        _lib.check(rc, "anyloc_vit_extract")
        return out


def resolve_state_dict(name, device):
    """Where the weights come from, in order: $ANYLOC_B200_WEIGHTS_DIR/<name>.pth (a plain upstream
    state_dict; for the timm names the timm checkpoint, which has the DINOv1 key names), the torch.hub
    checkpoint the reference itself loads (utilities.py:239-240, dino_extractor.py:82; needs network or
    a warm hub cache), or -- only when ANYLOC_B200_RANDOM_INIT=1 -- a seeded random init for synthetic
    benchmarks."""
    wdir = os.environ.get("ANYLOC_B200_WEIGHTS_DIR")
    if wdir:
        path = os.path.join(wdir, f"{name}.pth")
        if os.path.isfile(path):
            return torch.load(path, map_location="cpu")
    if os.environ.get("ANYLOC_B200_RANDOM_INIT") == "1":
        return random_state_dict(TIMM_ARCH.get(name, name), seed=int(os.environ.get("ANYLOC_B200_SEED", "0")),
                                 device=device)
    if name in TIMM_ARCH:
        raise _lib.AnylocError(
            f"cannot obtain weights for {name}: timm checkpoints are not downloaded by anyloc_b200. Put the timm "
            f"state_dict at $ANYLOC_B200_WEIGHTS_DIR/{name}.pth, or set ANYLOC_B200_RANDOM_INIT=1 for synthetic "
            "benchmarking")
    repo = "facebookresearch/dino:main" if ARCHS[name].family == "dino" else "facebookresearch/dinov2"
    try:
        model = torch.hub.load(repo, name)
    except Exception as e:  # offline box
        raise _lib.AnylocError(
            f"cannot obtain weights for {name}: torch.hub.load failed ({type(e).__name__}: {e}). Put an upstream "
            f"state_dict at $ANYLOC_B200_WEIGHTS_DIR/{name}.pth, or set ANYLOC_B200_RANDOM_INIT=1 for "
            "synthetic benchmarking") from e
    if hasattr(model, "state_dict"):
        return model.state_dict()
    return model
