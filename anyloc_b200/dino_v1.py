"""Drop-in mirror of DINOv1's `ViTExtractor` (/root/reference/dino_extractor.py:30-348), the extractor
behind AnyLoc's DINO (v1) results: same constructor, attributes and methods, with the forward run by the
CUDA ViT (`anyloc_vit_extract`, overlapping patch embedding at `stride`) and log-binning by
`anyloc_log_bin`.  CUDA only -- no CPU fallback.

Put `<repo>/anyloc_b200/dropin` first on PYTHONPATH to make `from dino_extractor import ViTExtractor` in
the reference's scripts resolve here (see INTEGRATION.md).
"""
import pathlib
from typing import List, Tuple, Union

import numpy as np
import torch

from . import _lib
from . import vit as _vit
from .utilities import _PrecisionPolicy, to_np


def log_bin(x: torch.Tensor, gh: int, gw: int, hierarchy: int = 2) -> torch.Tensor:
    """ViTExtractor._log_bin (dino_extractor.py:260-306) of a row-major grid of descriptors:
    x [B, gh*gw, C] fp32 on a CUDA device -> [B, gh*gw, 17*C] (bin-major: bin*C + c)."""
    if x.dim() != 3 or x.shape[1] != gh * gw:
        raise ValueError(f"expected [B, {gh}*{gw}, C] descriptors, got {tuple(x.shape)}")
    if not x.is_cuda:
        raise _lib.AnylocError("log_bin runs on CUDA devices only; there is no CPU fallback")
    x = x.to(torch.float32).contiguous()
    B, _, Cd = x.shape
    if Cd % 4:
        raise ValueError(f"descriptor dimension {Cd} must be a multiple of 4")
    out = torch.empty(B, gh * gw, 17 * Cd, device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        rc = _lib.load().anyloc_log_bin(_lib.ptr(x), B, gh, gw, Cd, hierarchy, _lib.ptr(out), _lib.stream_ptr())
    _lib.check(rc, "anyloc_log_bin")
    return out


class ViTExtractor(_PrecisionPolicy):
    """Extract DINOv1 descriptors (dino_extractor.py:30-348).

    Same constructor (`model_type`, `stride`, `model`, `device`), attributes (`model_type`, `device`, `p`,
    `stride` as a tuple, `mean`, `std`, `load_size`, `num_patches`) and methods (`preprocess`,
    `extract_descriptors`, `_extract_features`, `_log_bin`).  Models: dino_vits8 / vits16 / vitb8 / vitb16 and
    the timm names the reference maps onto them.  A passed `model` (nn.Module) supplies its state_dict; without
    one the weights come from vit.resolve_state_dict.  The forward stops at the hooked module, which is
    output-identical to the reference's full forward + hook.  Keyword-only `weights`, `gemm_engine` and
    `precision` as in DinoV2ExtractFeatures.  Attention maps (facet 'attn', extract_saliency_maps) are not
    provided: they need the full T x T probabilities, which the fused attention kernel never materialises."""

    def __init__(self, model_type: str = "dino_vits8", stride: int = 4, model=None, device: str = "cuda", *,
                 weights=None, gemm_engine: str = "auto", precision: str = None):
        arch_name = _vit.TIMM_ARCH.get(model_type, model_type)
        if arch_name not in _vit.ARCHS or _vit.ARCHS[arch_name].family != "dino":
            raise ValueError(f"unknown DINOv1 model_type {model_type!r}; expected one of "
                             f"{sorted(n for n, a in _vit.ARCHS.items() if a.family == 'dino') + sorted(_vit.TIMM_ARCH)}")
        self.model_type = model_type
        self.device = device
        self._arch = arch_name
        self.p = _vit.ARCHS[arch_name].patch
        s = tuple(stride) if isinstance(stride, (tuple, list)) else (stride, stride)
        assert all((self.p // s_) * s_ == self.p for s_ in s), f"stride {s} should divide patch_size {self.p}"
        if s[0] != s[1]:
            raise ValueError(f"stride {s}: only equal row and column strides are supported")
        self.stride = s
        self._dev = _lib.require_cuda(device)
        self.mean = (0.485, 0.456, 0.406) if "dino" in model_type else (0.5, 0.5, 0.5)
        self.std = (0.229, 0.224, 0.225) if "dino" in model_type else (0.5, 0.5, 0.5)
        if weights is None:
            weights = model.state_dict() if model is not None else _vit.resolve_state_dict(model_type, self._dev)
        self.gemm_engine = gemm_engine
        self._init_precision(precision, weights)
        self._feats = []
        self.hook_handlers = []
        self.load_size = None
        self.num_patches = None

    def _make_weights(self, state_dict, pair):
        return _vit.VitWeights(self._arch, state_dict, self._dev, pair=pair, stride=self.stride[0])

    def preprocess(self, image: Union[str, pathlib.Path, np.ndarray, torch.Tensor],
                   load_size: Union[int, Tuple[int, int]] = None):
        """dino_extractor.py:162-188 (host code): PIL LANCZOS resize (shorter side to an int load_size, or to
        (h, w)), then ToTensor + Normalize.  -> ([1,3,h,w] fp32 CPU tensor, PIL image)."""
        from PIL import Image
        if isinstance(image, (str, pathlib.Path)):
            pil_image = Image.open(image).convert("RGB")
        else:
            pil_image = Image.fromarray(to_np(image, np.uint8)).convert("RGB")
        if load_size is not None:
            w, h = pil_image.size
            if isinstance(load_size, int):           # torchvision Resize(int): shorter side -> load_size
                short, long = (w, h) if w <= h else (h, w)
                new_short, new_long = load_size, int(load_size * long / short)
                size = (new_short, new_long) if w <= h else (new_long, new_short)      # (w, h)
            else:
                size = (int(load_size[1]), int(load_size[0]))
            if size != (w, h):
                pil_image = pil_image.resize(size, Image.LANCZOS)
        x = torch.from_numpy(np.array(pil_image, dtype=np.uint8)).permute(2, 0, 1).float().div(255)
        mean = torch.tensor(self.mean, dtype=torch.float32)[:, None, None]
        std = torch.tensor(self.std, dtype=torch.float32)[:, None, None]
        return x.sub(mean).div(std)[None, ...], pil_image

    def _grid(self, H, W):
        return 1 + (H - self.p) // self.stride[0], 1 + (W - self.p) // self.stride[1]

    def _run(self, batch, layer, facet, include_cls, desc):
        if facet not in ("query", "key", "value", "token"):
            raise TypeError(f"{facet} is not a supported facet.")
        if not isinstance(batch, torch.Tensor) or batch.dim() != 4:
            raise ValueError("expected an image batch [B,3,H,W]")
        B, _, H, W = batch.shape
        if not 0 <= layer < self._vit.depth:
            raise IndexError(f"layer {layer} out of range for {self.model_type} with {self._vit.depth} blocks")
        with torch.no_grad():
            out = self._run_guarded(lambda m: m.extract(batch, layer, facet, include_cls, False, self.gemm_engine,
                                                        desc=desc))
        self.load_size = (H, W)
        self.num_patches = self._grid(H, W)
        return out

    def _extract_features(self, batch: torch.Tensor, layers: List[int] = 11, facet: str = "key") -> List[torch.Tensor]:
        """dino_extractor.py:240-258: a one-element list; q/k/v as [B,h,t,64], token as [B,t,d] (t includes CLS)."""
        if facet == "attn":
            raise _lib.AnylocError("facet 'attn' (T x T attention maps) is out of scope for anyloc_b200: the fused "
                                   "attention kernel never materialises the probabilities; it is used only for "
                                   "visualisation (scripts/dino_attention.py)")
        layer_list = [layers] if isinstance(layers, int) else list(layers)
        feats = []
        for layer in layer_list:
            x = self._run(batch, layer, facet, True, "plain")
            if facet != "token":
                B, t, D = x.shape
                x = x.reshape(B, t, D // 64, 64).permute(0, 2, 1, 3)
            feats.append(x)
        self._feats = feats
        return feats

    def _log_bin(self, x: torch.Tensor, hierarchy: int = 2) -> torch.Tensor:
        """dino_extractor.py:260-306 on a [B,h,t-1,d] feature map of the last extraction's grid -> [B,1,t-1,17*h*d]"""
        desc = x.to(self._dev).permute(0, 2, 3, 1).flatten(start_dim=-2)
        return log_bin(desc, self.num_patches[0], self.num_patches[1], hierarchy).unsqueeze(1)

    def extract_descriptors(self, batch: torch.Tensor, layer: int = 11, facet: str = "key", bin: bool = False,
                            include_cls: bool = False) -> torch.Tensor:
        """dino_extractor.py:308-332: [B,1,t,d'] fp32 on `device`, not normalised; q/k/v channels head-interleaved
        (c = dd*heads + head), token channels plain; CLS dropped unless include_cls; bin -> 17*d' log-binned."""
        assert facet in ["key", "query", "value", "token"], f"""{facet} is not a supported facet for descriptors.
                                                             choose from ['key' | 'query' | 'value' | 'token'] """
        if include_cls:
            assert not bin, "bin = True and include_cls = True are not supported together, set one of them False."
        x = self._run(batch, layer, facet, include_cls, "interleaved")
        if bin:
            x = log_bin(x, self.num_patches[0], self.num_patches[1])
        return x.unsqueeze(1)

    def extract_saliency_maps(self, batch: torch.Tensor) -> torch.Tensor:
        raise _lib.AnylocError("extract_saliency_maps is out of scope for anyloc_b200: it needs the T x T attention "
                               "probabilities of the last layer, which the fused attention kernel never materialises; "
                               "it is used only for visualisation (scripts/dino_attention.py)")
