"""TEST INFRASTRUCTURE -- CPU restatement of facebookresearch/dino @ main `vision_transformer.py`
(VisionTransformer, Block, Attention, Mlp, PatchEmbed), the DINOv1 models the reference's
ViTExtractor loads through torch.hub (/root/reference/dino_extractor.py:82) and hooks at
`blocks[l]`, `blocks[l].attn` and `blocks[l].attn.attn_drop` (:215-230).  The package is not
vendored by the reference and cannot be fetched here, so this file restates its published
forward pass:

  prepare_tokens: Conv2d(3,D,p,p) -> flatten -> cat cls -> + interpolate_pos_encoding(x, w, h)
     (w, h = the image's dim 2 and 3: rows and columns; identity when the grid has the pretrained
     number of cells and the image is square, else bicubic with scale_factor (g+0.1)/sqrt(N))
  block: y, attn = attn(norm1(x)); x += y;  x += mlp(norm2(x))      (no LayerScale)
  attn : softmax((q k^T) * 64**-0.5) -> attn_drop -> @ v -> proj; returns (x, attn)
  mlp  : fc2(GELU_erf(fc1(x)))
  LayerNorm eps 1e-6, qkv bias, mlp_ratio 4; init trunc_normal .02 for Linear, pos_embed and
  cls_token, zero bias, LayerNorm (1, 0).

Module and parameter names follow the upstream state_dict, so hub (and timm) weights load
unchanged and the reference's hooks and `patch_vit_resolution` (which sets
`patch_embed.proj.stride` and replaces `interpolate_pos_encoding`) run on it unmodified.
Cross-checked in tests against transformers' independent ViTModel.
"""
import math

import torch
from torch import nn

ARCHS = {
    # name: (embed_dim, depth, heads, patch)
    "dino_vits8": (384, 12, 6, 8),
    "dino_vits16": (384, 12, 6, 16),
    "dino_vitb8": (768, 12, 12, 8),
    "dino_vitb16": (768, 12, 12, 16),
}


class PatchEmbed(nn.Module):
    def __init__(self, img_size=224, patch_size=16, in_chans=3, embed_dim=768):
        super().__init__()
        self.img_size, self.patch_size = img_size, patch_size
        self.num_patches = (img_size // patch_size) * (img_size // patch_size)
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)

    def forward(self, x):
        return self.proj(x).flatten(2).transpose(1, 2)


class Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden, dim)
        self.drop = nn.Dropout(0.0)

    def forward(self, x):
        return self.drop(self.fc2(self.drop(self.act(self.fc1(x)))))


class Attention(nn.Module):
    def __init__(self, dim, num_heads):
        super().__init__()
        self.num_heads = num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.attn_drop = nn.Dropout(0.0)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(0.0)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
        q, k, v = qkv[0], qkv[1], qkv[2]
        attn = ((q @ k.transpose(-2, -1)) * self.scale).softmax(dim=-1)
        attn = self.attn_drop(attn)
        x = (attn @ v).transpose(1, 2).reshape(B, N, C)
        return self.proj_drop(self.proj(x)), attn


class Block(nn.Module):
    def __init__(self, dim, num_heads):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-6)
        self.attn = Attention(dim, num_heads)
        self.drop_path = nn.Identity()
        self.norm2 = nn.LayerNorm(dim, eps=1e-6)
        self.mlp = Mlp(dim, 4 * dim)

    def forward(self, x, return_attention=False):
        y, attn = self.attn(self.norm1(x))
        if return_attention:
            return attn
        x = x + self.drop_path(y)
        return x + self.drop_path(self.mlp(self.norm2(x)))


class VisionTransformer(nn.Module):
    def __init__(self, name="dino_vits8", depth_override=None):
        super().__init__()
        dim, depth, heads, patch = ARCHS[name]
        if depth_override is not None:
            depth = depth_override
        self.num_features = self.embed_dim = dim
        self.patch_embed = PatchEmbed(224, patch, 3, dim)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, self.patch_embed.num_patches + 1, dim))
        self.pos_drop = nn.Dropout(0.0)
        self.blocks = nn.ModuleList([Block(dim, heads) for _ in range(depth)])
        self.norm = nn.LayerNorm(dim, eps=1e-6)
        self.head = nn.Identity()
        nn.init.trunc_normal_(self.pos_embed, std=0.02)
        nn.init.trunc_normal_(self.cls_token, std=0.02)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.trunc_normal_(m.weight, std=0.02)
                if m.bias is not None:
                    nn.init.zeros_(m.bias)
            elif isinstance(m, nn.LayerNorm):
                nn.init.ones_(m.weight)
                nn.init.zeros_(m.bias)

    def interpolate_pos_encoding(self, x, w, h):
        npatch = x.shape[1] - 1
        N = self.pos_embed.shape[1] - 1
        if npatch == N and w == h:
            return self.pos_embed
        class_pos_embed = self.pos_embed[:, 0]
        patch_pos_embed = self.pos_embed[:, 1:]
        dim = x.shape[-1]
        w0 = w // self.patch_embed.patch_size
        h0 = h // self.patch_embed.patch_size
        w0, h0 = w0 + 0.1, h0 + 0.1
        patch_pos_embed = nn.functional.interpolate(
            patch_pos_embed.reshape(1, int(math.sqrt(N)), int(math.sqrt(N)), dim).permute(0, 3, 1, 2),
            scale_factor=(w0 / math.sqrt(N), h0 / math.sqrt(N)), mode="bicubic")
        assert int(w0) == patch_pos_embed.shape[-2] and int(h0) == patch_pos_embed.shape[-1]
        patch_pos_embed = patch_pos_embed.permute(0, 2, 3, 1).view(1, -1, dim)
        return torch.cat((class_pos_embed.unsqueeze(0), patch_pos_embed), dim=1)

    def prepare_tokens(self, x):
        B, nc, w, h = x.shape
        x = self.patch_embed(x)
        x = torch.cat((self.cls_token.expand(B, -1, -1), x), dim=1)
        x = x + self.interpolate_pos_encoding(x, w, h)
        return self.pos_drop(x)

    def forward(self, x):
        x = self.prepare_tokens(x)
        for blk in self.blocks:
            x = blk(x)
        return self.head(self.norm(x)[:, 0])


def build(name, seed=0, depth_override=None):
    """Random-init model with the upstream init recipe, deterministic in `seed` (CPU generator), eval mode."""
    g = torch.random.get_rng_state()
    torch.manual_seed(seed)
    m = VisionTransformer(name, depth_override=depth_override).eval()
    torch.random.set_rng_state(g)
    for p in m.parameters():
        p.requires_grad_(False)
    return m


def from_state_dict(sd, name, depth=None):
    """restated model holding exactly the tensors of `sd` (no random init)"""
    if depth is None:
        depth = 1 + max(int(k.split(".")[1]) for k in sd if k.startswith("blocks."))
    with torch.device("meta"):
        m = VisionTransformer(name, depth_override=depth)
    m.load_state_dict({k: v.detach().cpu().float() for k, v in sd.items()
                       if not k.startswith("blocks.") or int(k.split(".")[1]) < depth}, strict=False, assign=True)
    for p in m.parameters():
        p.requires_grad_(False)
    return m.eval()


def perturb(model, seed=1, scale=0.05):
    """Make biases / LayerNorm non-trivial so tests exercise them (upstream init leaves them at 0/1)."""
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if n.endswith("bias") or "norm" in n:
                p.add_(scale * torch.randn(p.shape, generator=gen))
        model.cls_token.add_(0.02 * torch.randn(model.cls_token.shape, generator=gen))
    return model


# ----------------------------------------------------------------- extractor oracle (independent restatement)
def pos_encoding(model, gh, gw, H, W):
    """[1, 1+gh*gw, D]: the table itself when the grid has the pretrained cell count and the image is square,
    else bicubic with scale (g+0.1)/sqrt(N) (align_corners=False, the given scale drives the coordinates)"""
    pos = model.pos_embed
    N = pos.shape[1] - 1
    if gh * gw == N and H == W:
        return pos
    m = int(math.sqrt(N))
    patch = nn.functional.interpolate(pos[:, 1:].reshape(1, m, m, -1).permute(0, 3, 1, 2),
                                      scale_factor=((gh + 0.1) / math.sqrt(N), (gw + 0.1) / math.sqrt(N)),
                                      mode="bicubic", align_corners=False, recompute_scale_factor=False)
    assert tuple(patch.shape[-2:]) == (gh, gw)
    return torch.cat([pos[:, :1], patch.permute(0, 2, 3, 1).reshape(1, gh * gw, -1)], dim=1)


def facet_tokens(model, img, stride, layer, facet):
    """[B, 1+gh*gw, D] fp32: block `layer`'s output (token) or its q/k/v projection in qkv column order
    (head*64 + dd), with the patch embedding at `stride`.  -> (tokens, (gh, gw))"""
    p = model.patch_embed.patch_size
    B, _, H, W = img.shape
    conv = model.patch_embed.proj
    x = nn.functional.conv2d(img, conv.weight, conv.bias, stride=stride)
    gh, gw = x.shape[-2:]
    x = torch.cat([model.cls_token.expand(B, -1, -1), x.flatten(2).transpose(1, 2)], dim=1)
    x = x + pos_encoding(model, gh, gw, H, W)
    for blk in model.blocks[:layer]:
        x = blk(x)
    blk = model.blocks[layer]
    if facet == "token":
        return blk(x), (gh, gw)
    D = x.shape[-1]
    i = {"query": 0, "key": 1, "value": 2}[facet]
    return blk.attn.qkv(blk.norm1(x))[..., i * D:(i + 1) * D], (gh, gw)


def interleave_heads(x, heads):
    """qkv column order (head*64 + dd) -> ViTExtractor's descriptor order (dd*heads + head)"""
    *lead, D = x.shape
    return x.reshape(*lead, heads, D // heads).transpose(-1, -2).reshape(*lead, D)


def log_bin(x, gh, gw):
    """hierarchy-2 log-binning of x [B, gh*gw, C] -> [B, gh*gw, 17*C]: bins 0-8 x at the 3x3 neighbours, 9-16 the
    3x3 average (count_include_pad=False) at the neighbours 3 cells away (centre skipped), coordinates clamped"""
    B, N, C = x.shape
    m = x.reshape(B, gh, gw, C).permute(0, 3, 1, 2)
    a1 = nn.functional.avg_pool2d(m, 3, stride=1, padding=1, count_include_pad=False)
    ys, xs = torch.arange(gh), torch.arange(gw)
    parts = []
    for src, step in ((m, 1), (a1, 3)):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                if step == 3 and dy == 0 and dx == 0:
                    continue
                iy, ix = (ys + step * dy).clamp(0, gh - 1), (xs + step * dx).clamp(0, gw - 1)
                parts.append(src[:, :, iy][:, :, :, ix])
    return torch.cat(parts, dim=1).flatten(2).transpose(1, 2)


def extract_descriptors(model, img, stride, layer=11, facet="key", bin=False, include_cls=False):
    """ViTExtractor.extract_descriptors semantics: [B, 1, t, d'] fp32, not normalised"""
    heads = model.blocks[0].attn.num_heads
    with torch.no_grad():
        x, (gh, gw) = facet_tokens(model, img.float(), stride, layer, facet)
        if facet != "token":
            x = interleave_heads(x, heads)
        if not include_cls:
            x = x[:, 1:]
        if bin:
            x = log_bin(x, gh, gw)
    return x.unsqueeze(1)
