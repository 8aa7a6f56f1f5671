"""Seeded inputs shared by the DINOv1 golden generator (tests/golden/make_golden_dino_v1.py) and the DINOv1 tests."""
import torch

from oracle import dino_v1_restated as d1

# tag: (model, stride, H, W, batch)
CASES = {
    "vits8_s4_60x76": ("dino_vits8", 4, 60, 76, 2),         # W not a multiple of the patch or the stride grid
    "vitb16_s8_64x64": ("dino_vitb16", 8, 64, 64, 1),
    "vits16_s16_48x64": ("dino_vits16", 16, 48, 64, 1),      # H != W: resampled even at the native stride
    "vits16_s8_120x120": ("dino_vits16", 8, 120, 120, 1),    # 14 x 14 grid of a square image: table passes through
}
LAYERS = (11, 5)
FACETS = ("query", "key", "value", "token")
LOG_BIN_GRIDS = ((1, 1), (1, 5), (2, 2), (3, 3), (5, 7))


def model_for(name):
    return d1.perturb(d1.build(name, seed=0), seed=1)


def image_for(tag):
    _, _, H, W, B = CASES[tag]
    return torch.randn(B, 3, H, W, generator=torch.Generator().manual_seed(sum(map(ord, tag))))


def log_bin_input(gh, gw, C=8, B=2):
    return torch.randn(B, gh * gw, C, generator=torch.Generator().manual_seed(100 * gh + gw))
