"""Drop-in mirror of the hot-path API of AnyLoc's `utilities.py`
(/root/reference/utilities.py): `DinoV2ExtractFeatures` (:219-288), `VLAD` (:624-1008),
`get_top_k_recall` (:390-469) plus the pass-through helpers the callers import from the same
module (`seed_everything` :505-519, `reduce_pca` :522-586, `CustomDataset` :25-74, `to_np`
:79-97).  Same names, argument meaning and error behaviour; the arithmetic runs in hand-written
sm_100a kernels behind the C ABI of include/anyloc_b200.h.  CUDA only -- no CPU fallback.

Put `<repo>/anyloc_b200/dropin` first on PYTHONPATH to make `from utilities import ...` in the
reference's scripts (scripts/dino_v2_vlad.py:37-38,50) resolve here (see INTEGRATION.md).
"""
import ctypes as C
import os
import random
from typing import List, Literal, Tuple, Union

import numpy as np
import torch

from . import _lib
from . import vit as _vit

_DINO_V2_MODELS = Literal["dinov2_vits14", "dinov2_vitb14", "dinov2_vitl14", "dinov2_vitg14"]
_DINO_FACETS = Literal["query", "key", "value", "token"]


# ------------------------------------------------------------------ helpers (pass-through)
class CustomDataset:
    """Abstract parent of the reference's custom datasets (utilities.py:25-74)."""

    def __init__(self) -> None:
        self.database_num = None
        self.queries_num = None
        self.soft_positives_per_query = None

    def get_image_paths(self):
        if hasattr(self, "images_paths"):
            return self.images_paths
        raise NotImplementedError("Not handled!")

    def get_positives(self):
        if hasattr(self, "soft_positives_per_query"):
            return self.soft_positives_per_query
        raise NotImplementedError("Not handled!")

    def get_image_relpaths(self, i: Union[int, List[int]]) -> Union[List[str], str]:
        single = type(i) == int
        paths = self.get_image_paths()
        depth = getattr(self, "_imgs_level", 2)
        rel = ["/".join(paths[k].split("/")[-depth:]) for k in ([i] if single else i)]
        return rel[0] if single else rel

    def __getitem__(self, index):
        raise NotImplementedError("Not created!")

    def __len__(self):
        if hasattr(self, "images_paths"):
            return len(self.get_image_paths())
        raise NotImplementedError("Not handled!")


def to_np(x, ret_type=float) -> np.ndarray:
    """utilities.py:79-97."""
    arr = x.detach().cpu().numpy() if type(x) == torch.Tensor else np.array(x)
    return arr.astype(ret_type)


def to_pil_list(x):
    """utilities.py:99-129: an image / batch ([B,C,H,W], [B,H,W,C], [C,H,W] or [H,W,C]) -> list of PIL images, each
    min-max normalised to 0..255.  Host-side helper (visualisation), not on the accelerated path."""
    from PIL import Image
    if type(x) == Image.Image or (type(x) == list and type(x[0]) == Image.Image):
        return x
    x = to_np(x)
    if len(x.shape) == 3:
        x = x[np.newaxis, ...]
    out = []
    for img in x:
        if img.shape[0] in [1, 3]:
            img = img.transpose(1, 2, 0)
        norm = (img - img.min()) / (img.max() - img.min())
        out.append(Image.fromarray((norm * 255).astype(np.uint8)))
    return out


def pad_img(img: np.ndarray, padding: int, color: tuple = (0, 0, 0)) -> np.ndarray:
    """utilities.py:474-500: [H,W,3] -> [H+2P, W+2P, 3] with an RGB border.  Host-side helper."""
    if type(color) == list:
        color = tuple(color)
    assert len(color) == 3, "Color should be (R, G, B) value"
    ret = np.ones((img.shape[0] + 2 * padding, img.shape[1] + 2 * padding, 3), np.uint8) * np.array(color)
    ret[padding:-padding, padding:-padding] = img
    return ret.astype(img.dtype)


def concat_desc_dists_clusters(cluster_centers: torch.Tensor, descs: torch.Tensor) -> torch.Tensor:
    """utilities.py:590-619: per descriptor, the unit residuals to every centre, concatenated and L2-normalised
    ([n, k*d]).  Plain tensor algebra on the caller's device, as in the reference (not on the hot path)."""
    assert type(cluster_centers) == type(descs) == torch.Tensor
    d = descs[:, None, :] - cluster_centers[None, ...]
    d = d / d.norm(dim=-1, keepdim=True)
    cat = d.reshape(d.shape[0], -1)
    return cat / cat.norm(dim=-1, keepdim=True)


def seed_everything(seed=42):
    """utilities.py:505-519."""
    random.seed(seed)
    os.environ["PYTHONHASHSEED"] = str(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False
    print(f"Seed set to: {seed} (type: {type(seed)})")


def _gemm_nt_dev(a, b, bias=None):
    """C = a @ b.T (+ bias) in fp32-equivalent precision on the tcgen05 engine (anyloc_gemm_nt, tf32 (hi,lo) pairs);
    a [M,K], b [N,K] device fp32, K padded to a multiple of 4 with zeros."""
    lib = _lib.load()
    pad = (-a.shape[1]) % 4
    if pad:
        a, b = torch.nn.functional.pad(a, (0, pad)), torch.nn.functional.pad(b, (0, pad))
    a, b = a.contiguous(), b.contiguous()
    M, K = a.shape
    N = b.shape[0]
    out = torch.empty(M, N, device=a.device, dtype=torch.float32)
    with torch.cuda.device(a.device):
        pairs = []
        for t in (a, b):
            hi, lo = torch.empty_like(t), torch.empty_like(t)
            _lib.check(lib.anyloc_split_tf32(_lib.ptr(t), _lib.ptr(hi), _lib.ptr(lo), t.numel(), _lib.stream_ptr()),
                       "anyloc_split_tf32")
            pairs += [hi, lo]
        rc = lib.anyloc_gemm_nt(_lib.ptr(pairs[0]), _lib.ptr(pairs[1]), K, _lib.ptr(pairs[2]), _lib.ptr(pairs[3]), K,
                                M, N, K, _lib.PAIR["tf32"], C.c_float(1.0), _lib.EPI["bias"], _lib.ptr(bias), None, None,
                                _lib.ptr(out), None, N, _lib.PAIR["tf32"], _lib.ENGINE["auto"], _lib.stream_ptr())
    _lib.check(rc, "anyloc_gemm_nt")
    return out


class _PcaDev:
    """`sklearn.decomposition.PCA(k, svd_solver="full", whiten=...)` as reduce_pca uses it (utilities.py:560-586), on
    the GPU: the fit is a one-off fp64 eigen-decomposition of the smaller Gram / covariance matrix (torch.linalg.eigh,
    i.e. cuSOLVER: plumbing), the projections -- the part that touches every descriptor -- run as GEMMs on this
    library's tcgen05 engine.  Component signs follow sklearn's `svd_flip(u_based_decision=False)`."""

    def __init__(self, n_components, whiten=False):
        self.n_components, self.whiten = int(n_components), bool(whiten)

    def fit(self, x):
        n, d = x.shape
        k = self.n_components
        if not 0 <= k <= min(n, d):
            raise ValueError(f"n_components={k} must be between 0 and min(n_samples, n_features)={min(n, d)} with "
                             "svd_solver='full'")
        self.mean_ = x.mean(dim=0)
        xd = (x - self.mean_).double()
        if n <= d:
            ev, u = torch.linalg.eigh(xd @ xd.T)
            ev, u = ev.flip(0).clamp_min(0), u.flip(1)
            s = ev.sqrt()
            vt = (u[:, :k].T @ xd) / s[:k, None].clamp_min(1e-300)
        else:
            ev, v = torch.linalg.eigh(xd.T @ xd)
            ev, v = ev.flip(0).clamp_min(0), v.flip(1)
            s = ev.sqrt()
            vt = v[:, :k].T.contiguous()
        sign = torch.sign(torch.gather(vt, 1, vt.abs().argmax(dim=1, keepdim=True)))
        sign[sign == 0] = 1
        self.components_ = (vt * sign).float().contiguous()
        self.singular_values_ = s[:k].float()
        self.explained_variance_ = (s[:k] ** 2 / (n - 1)).float()
        self.all_singular_values_ = s
        return self

    def transform(self, x):
        y = _gemm_nt_dev(x - self.mean_, self.components_)
        if self.whiten:
            scale = self.explained_variance_.sqrt()
            scale[scale < torch.finfo(scale.dtype).eps] = torch.finfo(scale.dtype).eps
            y = y / scale
        return y


def reduce_pca(train_descs: np.ndarray, test_descs: np.ndarray, lower_dim: int, low_factor: float = 0.0,
               fallback: int = 256, svd_solver: str = "full", whitening: bool = False) \
        -> Tuple[np.ndarray, np.ndarray]:
    """PCA projection fitted on the training set (utilities.py:522-586; scripts/dino_v2_vlad.py:357-369 reduces the
    database / query VLADs with it).  Same arguments and return types (numpy in -> numpy out, torch tensors accepted);
    the arithmetic runs on the GPU -- see _PcaDev.  `svd_solver` is accepted for signature compatibility: the result
    is the exact ("full") decomposition."""
    assert 0 <= low_factor <= 1
    as_np = type(train_descs) == np.ndarray
    dev = _lib.require_cuda(None)
    tr, te = _as_device_f32(train_descs, dev), _as_device_f32(test_descs, dev)

    def ret(a, b):
        return (a.cpu().numpy(), b.cpu().numpy()) if as_np else (a.cpu(), b.cpu())

    if low_factor == 0.0:
        pca = _PcaDev(lower_dim, whiten=whitening).fit(tr)
        return ret(pca.transform(tr), pca.transform(te))
    n_samples, n_components = tr.shape
    if n_samples < n_components:
        print(f"Too few samples, fallback to {fallback}d first")
        both = torch.cat((tr, te))
        both = _PcaDev(fallback).fit(both).transform(both)
        tr, te = both[:n_samples].contiguous(), both[n_samples:].contiguous()
    n_low = int(low_factor * lower_dim)
    n_top = lower_dim - n_low
    print(f"Up: {n_top}, Down: {n_low}")
    pca = _PcaDev(tr.shape[1]).fit(tr)
    basis = torch.cat((pca.components_[:n_top], pca.components_[-n_low:])).contiguous()
    return ret(_gemm_nt_dev(tr - pca.mean_, basis), _gemm_nt_dev(te - pca.mean_, basis))


# ------------------------------------------------------------------ image pre-processing (extension)
IMAGENET_MEAN = (0.485, 0.456, 0.406)       # dvgl_benchmark/datasets_ws.py:22
IMAGENET_STD = (0.229, 0.224, 0.225)


def center_crop_box(h: int, w: int, patch: int = 14) -> Tuple[int, int, int, int]:
    """(top, left, h_new, w_new) of `T.CenterCrop(((h // 14) * 14, (w // 14) * 14))`
    (scripts/dino_v2_vlad.py:174-176); torchvision places the window at int(round((h - h_new) / 2.0))."""
    h_new, w_new = (h // patch) * patch, (w // patch) * patch
    return int(round((h - h_new) / 2.0)), int(round((w - w_new) / 2.0)), h_new, w_new


_INTERP = {"bilinear": 0, "bicubic": 1}


def preprocess_images(imgs: Union[np.ndarray, torch.Tensor], mean=IMAGENET_MEAN, std=IMAGENET_STD,
                      patch: int = 14, device: Union[str, torch.device, None] = None,
                      resize: Union[Tuple[int, int], None] = None, interpolation: str = "bilinear") -> torch.Tensor:
    """uint8 RGB images [B,H,W,3] (or one [H,W,3]) -> the extractor's input [B,3,H',W'] on the GPU: the reference's
    `base_transform` (ToTensor + Normalize, dvgl_benchmark/datasets_ws.py:20-23), optionally the dataset loader's
    `T.functional.resize(img, resize)` (:233-235, `resize=(480, 640)` is the reference default, configs.py:141; or the
    demo's bicubic down-scaling, demo/anyloc_vlad_generate.py:165-177) and the centre crop to a multiple of the patch
    size (scripts/dino_v2_vlad.py:174-176) in ONE kernel.  Without `resize` the result is bit-identical to the
    torchvision pipeline; with it, antialiased bilinear / bicubic resampling as torchvision applies to tensors (fp32
    rounding differences only).  A quarter of the host->device bytes of sending normalised fp32 images."""
    if type(imgs) == np.ndarray:
        imgs = torch.from_numpy(imgs)
    if imgs.dtype != torch.uint8:
        raise TypeError(f"preprocess_images expects uint8 pixels, got {imgs.dtype}")
    if imgs.dim() == 3:
        imgs = imgs[None]
    if imgs.dim() != 4 or imgs.shape[-1] != 3:
        raise ValueError(f"preprocess_images expects [B,H,W,3], got {tuple(imgs.shape)}")
    if interpolation not in _INTERP:
        raise ValueError(f"interpolation must be one of {sorted(_INTERP)}, got {interpolation!r}")
    dev = _lib.require_cuda(imgs.device if imgs.is_cuda else (torch.device(device) if device is not None else None))
    x = imgs.to(dev, non_blocking=True).contiguous()
    B, H, W, _ = x.shape
    hr, wr = (H, W) if resize is None else (int(resize[0]), int(resize[1]))
    top, left, hc, wc = center_crop_box(hr, wr, patch)
    if hc == 0 or wc == 0:
        raise ValueError(f"image {hr}x{wr} is smaller than one {patch}x{patch} patch")
    out = torch.empty(B, 3, hc, wc, device=dev, dtype=torch.float32)
    m3 = (C.c_float * 3)(*[float(v) for v in mean])
    s3 = (C.c_float * 3)(*[float(v) for v in std])
    with torch.cuda.device(dev):
        if resize is None:
            _lib.check(_lib.load().anyloc_preprocess_u8(_lib.ptr(x), B, H, W, top, left, hc, wc, m3, s3, _lib.ptr(out),
                                                        _lib.stream_ptr()), "anyloc_preprocess_u8")
        else:
            _lib.check(_lib.load().anyloc_preprocess_resize_u8(_lib.ptr(x), B, H, W, hr, wr, _INTERP[interpolation], top,
                                                               left, hc, wc, m3, s3, _lib.ptr(out), _lib.stream_ptr()),
                       "anyloc_preprocess_resize_u8")
    return out


# ------------------------------------------------------------------ extractor
class _HookHandle:
    def remove(self):
        pass


class _PrecisionPolicy:
    """How an extractor feeds fp32 operands to the tensor cores, shared by DinoV2ExtractFeatures and the DINOv1
    ViTExtractor (anyloc_b200/dino_v1.py): "tf32x3", "f16x3" or "auto" (see DinoV2ExtractFeatures).  Subclasses
    provide `_make_weights(state_dict, pair)` -> vit.VitWeights and run every forward through `_run_guarded`."""

    _OVERFLOW_MSG = ("f16x3 precision overflowed the fp16 operand range (|8*x| > 65504 somewhere in the network); "
                     "construct the extractor with precision='tf32x3' (or 'auto')")

    def _init_precision(self, precision, state_dict):
        precision = precision or os.environ.get("ANYLOC_B200_PRECISION", "auto")
        if precision not in ("tf32x3", "f16x3", "auto"):
            raise ValueError(f"precision must be 'auto', 'tf32x3' or 'f16x3', got {precision!r}")
        self._auto = precision == "auto"
        self._state_dict = state_dict if self._auto else None     # kept for the tf32x3 re-upload on an overflow
        self.precision = "f16x3" if self._auto else precision
        self._vit = self._make_weights(state_dict, "f16" if self.precision == "f16x3" else "tf32")
        # fp16-range guard of the f16x3 format: "sync" = checked before a call returns (one host sync per call),
        # "deferred" = the flag of call i is read at call i+1 / raise_if_overflowed() (no sync on the hot loop),
        # "off".  precision="auto" always checks synchronously (it has to decide before returning).
        self.check_finite = os.environ.get("ANYLOC_B200_CHECK_FINITE", "sync")
        if self.check_finite in ("1", "0"):
            self.check_finite = "sync" if self.check_finite == "1" else "off"
        self._pending_flag = None

    def raise_if_overflowed(self):
        """Deferred mode: reads the finite-flag of the last call (one host sync)."""
        flag, self._pending_flag = self._pending_flag, None
        if flag is not None and not bool(flag):
            raise _lib.AnylocError(self._OVERFLOW_MSG)

    def _switch_to_tf32(self):
        print("anyloc_b200: f16x3 operands overflowed the fp16 range -- switching this extractor to tf32x3 "
              "(full fp32 exponent range, ~2x slower)")
        self._vit = None
        torch.cuda.empty_cache()
        self._vit = self._make_weights(self._state_dict, "tf32")
        self.precision, self._auto, self._state_dict = "tf32x3", False, None

    def _run_guarded(self, run):
        """run(VitWeights) -> device tensor, checked against the fp16 range as configured"""
        if self.check_finite == "deferred" and not self._auto:
            self.raise_if_overflowed()
        out = run(self._vit)
        if self.precision != "f16x3" or (self.check_finite == "off" and not self._auto):
            return out
        flag = torch.isfinite(out).all()
        if self.check_finite == "deferred" and not self._auto:
            self._pending_flag = flag
            return out
        if bool(flag):
            return out
        if not self._auto:
            raise _lib.AnylocError(self._OVERFLOW_MSG)
        self._switch_to_tf32()
        return run(self._vit)


class DinoV2ExtractFeatures(_PrecisionPolicy):
    """Extract features from an intermediate layer of DINOv2 (utilities.py:219-288).

    Same constructor and call signature.  The forward stops at the hooked module (blocks
    0..layer-1, then either the whole block `layer` ("token") or norm1 + the requested third of
    its qkv projection), which is output-identical to the reference's full forward + hook.
    Extra keyword-only arguments: `weights` (an upstream state_dict, else see
    vit.resolve_state_dict), `gemm_engine` ("auto" | "tc3" | "simt") and `precision`: how fp32
    operands are fed to the tensor cores -- "tf32x3" (tf32 (hi,lo) pairs, full fp32 exponent range),
    "f16x3" (fp16 (hi,lo) pairs with power-of-two scaling: same ~22-bit products on the 2x faster
    kind::f16 path; operands beyond the fp16 range overflow to inf/NaN instead of losing accuracy
    silently, and the call raises) or "auto" (the default: f16x3 until a call overflows, then that
    call is redone and the extractor stays in tf32x3 -- trained DINOv2 checkpoints have outlier
    activations that random-init weights do not).  All accumulate in fp32 with round-to-nearest
    chunk accumulation."""

    def __init__(self, dino_model: _DINO_V2_MODELS, layer: int, facet: _DINO_FACETS = "token",
                 use_cls=False, norm_descs=True, device: str = "cpu", *, weights=None,
                 gemm_engine: str = "auto", precision: str = None) -> None:
        self.vit_type: str = dino_model
        self.device = torch.device(device)
        self._dev = _lib.require_cuda(self.device)
        if facet not in _lib.FACET:
            raise ValueError(f"facet must be one of {sorted(_lib.FACET)}, got {facet!r}")
        sd = weights if weights is not None else _vit.resolve_state_dict(dino_model, self._dev)
        self.layer: int = layer
        self._init_precision(precision, sd)
        self.facet = facet
        self.use_cls = use_cls
        self.norm_descs = norm_descs
        self.gemm_engine = gemm_engine
        self.fh_handle = _HookHandle()
        self._hook_out = None

    @property
    def dino_model(self):
        """the device-resident backbone (vit.VitWeights)"""
        return self._vit

    def _make_weights(self, state_dict, pair):
        # only blocks 0..layer are ever executed (early exit), so only those are uploaded
        return _vit.VitWeights(self.vit_type, state_dict, self._dev, depth=self.layer + 1, pair=pair)

    def __call__(self, img: torch.Tensor) -> torch.Tensor:
        with torch.no_grad():
            return self._run_guarded(lambda m: m.extract(img, self.layer, self.facet, self.use_cls, self.norm_descs,
                                                         self.gemm_engine))

    def __del__(self):
        pass


# ------------------------------------------------------------------ VLAD
def _as_device_f32(x, device):
    if type(x) == np.ndarray:
        x = torch.from_numpy(x)
    return x.detach().to(device=device, dtype=torch.float32).contiguous()


def _normalize_rows_dev(x):
    """F.normalize(x) of a device matrix [R,D] (utilities.py:782-783)."""
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().anyloc_l2_normalize_rows(_lib.ptr(x), x.shape[0], x.shape[1], x.shape[1],
                                                        _lib.ptr(y), _lib.stream_ptr()), "l2_normalize_rows")
    return y


class _KMeans:
    """GPU stand-in for `fast_pytorch_kmeans.KMeans` as the reference uses it (utilities.py:766,
    :772, :786-787, :849): `.centroids`, `.fit(X)`, `.predict(X)`; cosine / euclidean similarity,
    numpy-seeded random-choice init, <=100 Lloyd iterations, tol 1e-4."""

    def __init__(self, n_clusters, max_iter=100, tol=1e-4, verbose=0, mode="euclidean", minibatch=None):
        if mode not in _lib.DIST:
            raise NotImplementedError(mode)
        self.n_clusters, self.max_iter, self.tol, self.mode = n_clusters, max_iter, tol, mode
        self.verbose, self.minibatch = verbose, minibatch
        self.centroids = None

    def _assign(self, x, centers):
        lib = _lib.load()
        R, D = x.shape
        K = centers.shape[0]
        labels = torch.empty(R, dtype=torch.int32, device=x.device)
        with torch.cuda.device(x.device):
            ws = _lib.workspaces.get(x.device, lib.anyloc_vlad_workspace_bytes(1, R, D, K), "kmeans")
            _lib.check(lib.anyloc_vlad_assign(_lib.ptr(x), _lib.ptr(centers), R, D, K, _lib.DIST[self.mode],
                                              _lib.ptr(labels), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
                       "anyloc_vlad_assign")
        return labels

    def _update(self, x, labels, c):
        """one Lloyd centroid update (anyloc_kmeans_update) -> (new centres, sum of squared centre shifts as a device
        tensor -- or a float, from a synchronous implementation)"""
        lib = _lib.load()
        n, D = x.shape
        K = c.shape[0]
        new_c = torch.empty_like(c)
        err = torch.zeros(1, device=x.device)
        with torch.cuda.device(x.device):
            ws = _lib.workspaces.get(x.device, lib.anyloc_kmeans_workspace_bytes(n, D, K), "kmeans_upd")
            _lib.check(lib.anyloc_kmeans_update(_lib.ptr(x), _lib.ptr(labels), _lib.ptr(c), n, D, K,
                                                _lib.ptr(new_c), _lib.ptr(err), _lib.ptr(ws), ws.numel(),
                                                _lib.stream_ptr()), "anyloc_kmeans_update")
        return new_c, err              # err stays on the device: fit_predict reads it one iteration late

    def predict(self, X):
        dev = _lib.require_cuda(X.device if isinstance(X, torch.Tensor) and X.is_cuda else None)
        was_cpu = not (isinstance(X, torch.Tensor) and X.is_cuda)
        labels = self._assign(_as_device_f32(X, dev), _as_device_f32(self.centroids, dev)).to(torch.int64)
        return labels.cpu() if was_cpu else labels

    def fit_predict(self, X, centroids=None):
        dev = _lib.require_cuda(X.device if X.is_cuda else None)
        was_cpu = not X.is_cuda
        x = _as_device_f32(X, dev)
        n, D = x.shape
        K = self.n_clusters
        if centroids is None:
            init = np.random.choice(n, size=[K], replace=False)      # numpy RNG, as upstream
            c = x[torch.from_numpy(init).to(dev)].contiguous()
        else:
            c = _as_device_f32(centroids, dev)
        # Lloyd iterations without a host sync on the critical path: iteration i+1 is enqueued BEFORE the convergence
        # test of iteration i is read (its error travels to pinned host memory behind an event), so the device never
        # idles on the host; when iteration i turns out to have converged, the speculative iteration is simply dropped
        # -- centres and labels are exactly those of the synchronous loop (fpk: break after the update whose shift <= tol)
        labels, pending = None, None            # pending = (labels_i, c_{i+1}, host error, event) of the previous iteration
        hosts = None
        for it in range(self.max_iter):
            labels_i = self._assign(x, c)
            c_next, err = self._update(x, labels_i, c)
            if not isinstance(err, torch.Tensor):                 # synchronous implementation (tests' CPU double)
                labels, c = labels_i, c_next
                if err <= self.tol:
                    break
                continue
            if hosts is None:
                hosts = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
            host = hosts[it & 1]
            host.copy_(err, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            if pending is not None:
                pending[3].synchronize()
                if float(pending[2][0]) <= self.tol:               # the PREVIOUS iteration had converged
                    labels, c = pending[0], pending[1]
                    pending = None
                    break
            pending = (labels_i, c_next, host, ev)
            labels, c = labels_i, c_next
        if pending is not None:
            pending[3].synchronize()                               # results of the last enqueued iteration are final
        self.centroids = c.cpu() if was_cpu else c
        labels = labels.to(torch.int64)
        return labels.cpu() if was_cpu else labels

    def fit(self, X, centroids=None):
        self.fit_predict(X, centroids)


VLAD_KERNEL_DESCRIPTION = ("VLAD v3.1: vlad_assign_tc_kernel (TMA stream + tcgen05 coarse scores + row norms + exact "
                           "re-scoring of the ambiguous rows by dedicated warps, wave-balanced tiles) -> "
                           "vlad_accumulate3_kernel (label-sorted residual sums + fused normalisation); prepared "
                           "vocabulary, 2 launches")


class VLAD:
    """Hard- and soft-assignment VLAD with the reference's constructor and methods (utilities.py:624-1008).

    `generate` / `generate_multi` take what the reference takes (CPU tensors / numpy arrays /
    ragged lists) and return what it returns (CPU tensors); CUDA tensors are also accepted and
    then stay on the device (the batched fast path).  The on-disk caches are honoured in the
    reference's own file formats: the vocabulary (`c_centers.pt`), and per image the labels
    (`<id>_l.pt`) / soft assignment (`<id>_s.pt`) and residual tensor (`<id>_r.pt`) are READ when
    present; labels / soft assignments are written like the reference does, the residual tensor
    (>=100 MB per image at ViT-G, K=32) only when `self.cache_residuals = True` or through
    `generate_res_vec(..., cache_id)`.  `vlad_mode="soft"` follows the reference's soft branch
    (:862-887), including its summation over the residuals to all centres."""

    def __init__(self, num_clusters: int, desc_dim: Union[int, None] = None, intra_norm: bool = True,
                 norm_descs: bool = True, dist_mode: str = "cosine", vlad_mode: str = "hard",
                 soft_temp: float = 1.0, cache_dir: Union[str, None] = None) -> None:
        self.num_clusters = num_clusters
        self.desc_dim = desc_dim
        self.intra_norm = intra_norm
        self.norm_descs = norm_descs
        self.mode = dist_mode
        self.vlad_mode = str(vlad_mode).lower()
        assert self.vlad_mode in ["soft", "hard"]
        self.soft_temp = soft_temp
        self.c_centers = None
        self.kmeans = None
        self._centers_dev = {}
        self._prepared_dev = None
        self.cache_residuals = False     # extension: write `<id>_r.pt` like the reference (104 MB per image at c2)
        self.cache_dir = cache_dir
        if self.cache_dir is not None:
            self.cache_dir = os.path.abspath(os.path.expanduser(self.cache_dir))
            if not os.path.exists(self.cache_dir):
                os.makedirs(self.cache_dir)
                print(f"Created cache directory: {self.cache_dir}")
            else:
                print(f"Warning: Cache directory already exists: {self.cache_dir}")
        else:
            print("VLAD caching is disabled.")

    # -- cache predicates (utilities.py:688-746)
    def can_use_cache_vlad(self):
        if self.cache_dir is None or not os.path.exists(self.cache_dir):
            return False
        return os.path.exists(f"{self.cache_dir}/c_centers.pt")

    def can_use_cache_ids(self, cache_ids: Union[List[str], str, None], only_residuals: bool = False) -> bool:
        if not self.can_use_cache_vlad() or cache_ids is None:
            return False
        if isinstance(cache_ids, str):
            cache_ids = [cache_ids]
        suffix = "l" if self.vlad_mode == "hard" else "s"
        for cid in cache_ids:
            if not os.path.exists(f"{self.cache_dir}/{cid}_r.pt"):
                return False
            if not only_residuals and not os.path.exists(f"{self.cache_dir}/{cid}_{suffix}.pt"):
                return False
        return True

    # -- vocabulary (utilities.py:749-791)
    def fit(self, train_descs: Union[np.ndarray, torch.Tensor, None]):
        self.kmeans = _KMeans(self.num_clusters, mode=self.mode)
        self._centers_dev = {}
        self._prepared_dev = None
        if self.can_use_cache_vlad():
            print("Using cached cluster centers")
            self.c_centers = torch.load(f"{self.cache_dir}/c_centers.pt")
            self.kmeans.centroids = self.c_centers
            if self.desc_dim is None:
                self.desc_dim = self.c_centers.shape[1]
                print(f"Desc dim set to {self.desc_dim}")
            return
        if train_descs is None:
            raise ValueError("No training descriptors given")
        if type(train_descs) == np.ndarray:
            train_descs = torch.from_numpy(train_descs).to(torch.float32)
        if self.desc_dim is None:
            self.desc_dim = train_descs.shape[1]
        dev = _lib.require_cuda(train_descs.device if train_descs.is_cuda else None)
        was_cpu = not train_descs.is_cuda
        x = _as_device_f32(train_descs, dev)
        if self.norm_descs:
            x = _normalize_rows_dev(x)
        self.kmeans.fit(x)
        self.c_centers = self.kmeans.centroids.cpu() if was_cpu else self.kmeans.centroids
        self.kmeans.centroids = self.c_centers
        if self.cache_dir is not None:
            print("Caching cluster centers")
            torch.save(self.c_centers.cpu(), f"{self.cache_dir}/c_centers.pt")

    def fit_and_generate(self, train_descs: Union[np.ndarray, torch.Tensor]) -> torch.Tensor:
        if type(train_descs) == np.ndarray:
            train_descs = torch.from_numpy(train_descs).to(torch.float32)
        self.fit(train_descs.reshape(-1, train_descs.shape[-1]))
        return self.generate_multi(train_descs)

    # -- device plumbing
    def _centers_on(self, dev):
        cc = self.c_centers
        key = (dev.index, id(cc), getattr(cc, "_version", None), cc.data_ptr() if isinstance(cc, torch.Tensor) else None)
        if key not in self._centers_dev:
            self._centers_dev = {key: _as_device_f32(self.c_centers, dev)}
        return self._centers_dev[key]

    def _prepared_on(self, dev, centers):
        """Device blob of anyloc_vlad_prepare for the current vocabulary (recomputed when c_centers is replaced or
        modified in place, or the distance mode changes)."""
        cc = self.c_centers
        key = (dev.index, id(cc), getattr(cc, "_version", None), self.mode, centers.data_ptr())
        cache = getattr(self, "_prepared_dev", None)
        if cache is None or cache[0] != key:
            lib = _lib.load()
            K, D = centers.shape
            blob = torch.empty(lib.anyloc_vlad_prepared_bytes(D, K), dtype=torch.uint8, device=dev)
            with torch.cuda.device(dev):
                _lib.check(lib.anyloc_vlad_prepare(_lib.ptr(centers), D, K, _lib.DIST[self.mode], _lib.ptr(blob),
                                                   blob.numel(), _lib.stream_ptr()), "anyloc_vlad_prepare")
            self._prepared_dev = cache = (key, blob)
        return cache[1]

    def _run(self, feats, n_valid, dev, want_labels=False):
        """feats [B,N,D] device fp32; n_valid [B] int32 device or None -> ([B,K*D], labels|None)
        (soft mode: the [B,N,K] assignment probabilities take the place of the labels)."""
        assert self.kmeans is not None
        assert self.c_centers is not None
        lib = _lib.load()
        B, N, D = feats.shape
        K = self.num_clusters
        centers = self._centers_on(dev)
        if centers.shape != (K, D):
            raise ValueError(f"cluster centres {tuple(centers.shape)} do not match K={K}, D={D}")
        out = torch.empty(B, K * D, device=dev, dtype=torch.float32)
        labels = torch.empty(B, N, device=dev, dtype=torch.int32) if want_labels else None
        if self.vlad_mode == "soft":        # utilities.py:862-887
            assign = torch.empty(B, N, K, device=dev, dtype=torch.float32) if want_labels else None
            with torch.cuda.device(dev):
                ws = _lib.workspaces.get(dev, lib.anyloc_vlad_workspace_bytes(B, N, D, K), "vlad")
                rc = lib.anyloc_vlad_generate_soft(_lib.ptr(feats), _lib.ptr(n_valid), _lib.ptr(centers), B, N, D, K,
                                                   float(self.soft_temp), int(bool(self.norm_descs)),
                                                   int(bool(self.intra_norm)), _lib.ptr(out), _lib.ptr(assign),
                                                   _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
            _lib.check(rc, "anyloc_vlad_generate_soft")
            return out, assign
        with torch.cuda.device(dev):
            ws = _lib.workspaces.get(dev, lib.anyloc_vlad_workspace_bytes(B, N, D, K), "vlad")
            prep = self._prepared_on(dev, centers)
            rc = lib.anyloc_vlad_generate_prepared(_lib.ptr(feats), _lib.ptr(n_valid), _lib.ptr(centers), _lib.ptr(prep),
                                                   prep.numel(), B, N, D, K, _lib.DIST[self.mode],
                                                   int(bool(self.norm_descs)), int(bool(self.intra_norm)),
                                                   _lib.ptr(out), _lib.ptr(labels), _lib.ptr(ws), ws.numel(),
                                                   _lib.stream_ptr())
        _lib.check(rc, "anyloc_vlad_generate_prepared")
        return out, labels

    # -- per-image cache (utilities.py:843-852 labels, :864-878 soft assignment, :951-970 residuals)
    def _cache_path(self, cache_id, suffix):
        return f"{self.cache_dir}/{cache_id}_{suffix}.pt"

    def _cache_active(self, cache_id):
        return cache_id is not None and self.can_use_cache_vlad()

    def _residuals_dev(self, x, dev):
        """x [N,D] device fp32 -> residual tensor [N,K,D] on the device (anyloc_vlad_residuals)."""
        centers = self._centers_on(dev)
        N, D = x.shape
        K = centers.shape[0]
        if centers.shape[1] != D:
            raise ValueError(f"cluster centres {tuple(centers.shape)} do not match descriptor dim {D}")
        out = torch.empty(N, K, D, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            _lib.check(_lib.load().anyloc_vlad_residuals(_lib.ptr(x), _lib.ptr(centers), N, D, K,
                                                         int(bool(self.norm_descs)), _lib.ptr(out), _lib.stream_ptr()),
                       "anyloc_vlad_residuals")
        return out

    def _from_residuals_dev(self, resid, labels, assign, dev):
        """descriptor [K*D] (device) of one image from its residual tensor + hard labels | soft assignment"""
        lib = _lib.load()
        N, K, D = resid.shape
        out = torch.empty(K * D, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            ws = _lib.workspaces.get(dev, lib.anyloc_vlad_from_residuals_workspace_bytes(D, K), "vlad_cache")
            _lib.check(lib.anyloc_vlad_from_residuals(_lib.ptr(resid), _lib.ptr(labels), _lib.ptr(assign), N, D, K,
                                                      int(bool(self.intra_norm)), _lib.ptr(out), _lib.ptr(ws),
                                                      ws.numel(), _lib.stream_ptr()), "anyloc_vlad_from_residuals")
        return out

    def _generate_cached(self, query_descs, cache_id, dev):
        """The reference's cache-aware path, file for file: residuals from `<id>_r.pt` when present (else computed
        from the features; written back only when `self.cache_residuals`), labels from `<id>_l.pt` / soft assignment
        from `<id>_s.pt` when present (else computed AND saved, like the reference).  Files are CPU tensors in the
        reference's own format, so a directory populated by either implementation serves both.  -> [K*D] device."""
        suffix = "l" if self.vlad_mode == "hard" else "s"
        have_r = os.path.isfile(self._cache_path(cache_id, "r"))
        have_a = os.path.isfile(self._cache_path(cache_id, suffix))
        x = None
        if query_descs is not None:
            x = _as_device_f32(query_descs, dev)
        elif not (have_r and have_a):
            raise ValueError(f"no descriptors given and the cache of {cache_id!r} is incomplete")
        if not have_r and not have_a and not getattr(self, "cache_residuals", False):
            # nothing cached yet: the fused fast path, keeping the assignment for the next run
            out, assign = self._run(x.unsqueeze(0), None, dev, want_labels=True)
            self._save_assignment(cache_id, suffix, assign[0])
            return out[0]
        if have_r:
            resid = torch.load(self._cache_path(cache_id, "r")).to(device=dev, dtype=torch.float32).contiguous()
        else:
            resid = self._residuals_dev(x, dev)
            if getattr(self, "cache_residuals", False):
                cid_dir = f"{self.cache_dir}/{os.path.split(cache_id)[0]}"
                if not os.path.isdir(cid_dir):
                    os.makedirs(cid_dir)
                    print(f"Created directory: {cid_dir}")
                torch.save(resid.cpu(), self._cache_path(cache_id, "r"))
        if have_a:
            assign = torch.load(self._cache_path(cache_id, suffix)).to(dev)
        else:
            _, assign = self._run(x.unsqueeze(0), None, dev, want_labels=True)
            assign = assign[0]
            self._save_assignment(cache_id, suffix, assign)
        if self.vlad_mode == "hard":
            return self._from_residuals_dev(resid, assign.to(torch.int32).contiguous(), None, dev)
        return self._from_residuals_dev(resid, None, assign.to(torch.float32).contiguous(), dev)

    def _save_assignment(self, cache_id, suffix, assign):
        cid_dir = f"{self.cache_dir}/{os.path.split(cache_id)[0]}"
        if not os.path.isdir(cid_dir):
            os.makedirs(cid_dir)
            print(f"Created directory: {cid_dir}")
        # the reference stores kmeans.predict's int64 labels / the fp32 [q, c] soft assignment, on the CPU
        a = assign.to(torch.int64) if suffix == "l" else assign
        torch.save(a.cpu(), self._cache_path(cache_id, suffix))

    # -- descriptors (utilities.py:819-926)
    def generate(self, query_descs: Union[np.ndarray, torch.Tensor, None], cache_id: Union[str, None] = None) \
            -> torch.Tensor:
        on_dev = isinstance(query_descs, torch.Tensor) and query_descs.is_cuda
        dev = _lib.require_cuda(query_descs.device if on_dev else None)
        if self._cache_active(cache_id):
            out = self._generate_cached(query_descs, cache_id, dev)
            return out if on_dev else out.cpu()
        x = _as_device_f32(query_descs, dev)
        out, _ = self._run(x.unsqueeze(0), None, dev)
        return out[0] if on_dev else out[0].cpu()

    def generate_multi(self, multi_query: Union[np.ndarray, torch.Tensor, list],
                       cache_ids: Union[List[str], None] = None) -> Union[torch.Tensor, list]:
        if cache_ids is not None and self.can_use_cache_vlad() and any(c is not None for c in cache_ids):
            # cache-aware: image by image like the reference (:917-918); `multi_query` may be [None] * n when
            # can_use_cache_ids() said the cache is complete (scripts/dino_v2_vlad.py:224-228)
            res = [self.generate(q, c) for (q, c) in zip(multi_query, cache_ids)]
            return torch.stack(res)
        if isinstance(multi_query, (list, tuple)):
            if len(multi_query) == 0:
                return torch.stack([])      # same failure as the reference on an empty list
            on_dev = all(isinstance(q, torch.Tensor) and q.is_cuda for q in multi_query)
            dev = _lib.require_cuda(multi_query[0].device if on_dev else None)
            qs = [_as_device_f32(q, dev) for q in multi_query]
            n_max = max(q.shape[0] for q in qs)
            D = qs[0].shape[1]
            feats = torch.zeros(len(qs), n_max, D, device=dev, dtype=torch.float32)
            for i, q in enumerate(qs):
                feats[i, :q.shape[0]] = q
            n_valid = torch.tensor([q.shape[0] for q in qs], dtype=torch.int32, device=dev)
            out, _ = self._run(feats, n_valid, dev)
            return out if on_dev else out.cpu()
        was_np = type(multi_query) == np.ndarray
        on_dev = isinstance(multi_query, torch.Tensor) and multi_query.is_cuda
        dev = _lib.require_cuda(multi_query.device if on_dev else None)
        if not on_dev and not was_np and multi_query.numel() * 4 > self._host_chunk_bytes:
            # large host batches (the driver hands over [n_imgs, n_patches, D] on the CPU): stream chunks
            step = max(1, self._host_chunk_bytes // (multi_query[0].numel() * 4))
            return torch.cat([self._run(_as_device_f32(multi_query[i:i + step], dev), None, dev)[0].cpu()
                              for i in range(0, multi_query.shape[0], step)])
        out, _ = self._run(_as_device_f32(multi_query, dev), None, dev)
        return out if on_dev else out.cpu()

    _host_chunk_bytes = 1 << 30

    # -- residual tensors (utilities.py:928-1008)
    def generate_res_vec(self, query_descs: Union[np.ndarray, torch.Tensor],
                         cache_id: Union[str, None] = None) -> torch.Tensor:
        assert self.kmeans is not None
        assert self.c_centers is not None
        if self._cache_active(cache_id) and os.path.isfile(self._cache_path(cache_id, "r")):
            return torch.load(self._cache_path(cache_id, "r"))
        on_dev = isinstance(query_descs, torch.Tensor) and query_descs.is_cuda
        dev = _lib.require_cuda(query_descs.device if on_dev else None)
        resid = self._residuals_dev(_as_device_f32(query_descs, dev), dev)
        resid = resid if on_dev else resid.cpu()
        if self._cache_active(cache_id):           # explicit request for the residual tensor: cache it as the reference does
            cid_dir = f"{self.cache_dir}/{os.path.split(cache_id)[0]}"
            if not os.path.isdir(cid_dir):
                os.makedirs(cid_dir)
                print(f"Created directory: {cid_dir}")
            torch.save(resid.cpu(), self._cache_path(cache_id, "r"))
        return resid

    def generate_multi_res_vec(self, multi_query: Union[np.ndarray, torch.Tensor, list],
                               cache_ids: Union[List[str], None] = None) -> Union[torch.Tensor, list]:
        if cache_ids is None:
            cache_ids = [None] * len(multi_query)
        res = [self.generate_res_vec(q, c) for (q, c) in zip(multi_query, cache_ids)]
        try:
            return torch.stack(res)
        except (TypeError, RuntimeError):
            return res              # ragged inputs stay a list


# ------------------------------------------------------------------ sibling aggregators (extension)
_POOL = {"average": 0, "avg": 0, "mean": 0, "max": 1, "gem": 2}


def pool_descriptors(patch_descs: torch.Tensor, method: str = "gem", gem_p: float = 3.0,
                     gem_use_abs: bool = False) -> torch.Tensor:
    """Global descriptors [N, d_dim] from patch features [N, n_p, d_dim] the way the reference's other DINOv2
    scripts pool them: `get_gem_descriptors` (scripts/dino_v2_gem.py:170-189; `gem_p`, `gem_use_abs`) and the
    "average" / "max" pooling of scripts/dino_v2_gp.py:130-135.  CPU in -> CPU out, CUDA in -> CUDA out."""
    if method not in _POOL:
        raise NotImplementedError(f"ID: {method}")          # scripts/dino_v2_gp.py:134-135
    assert len(patch_descs.shape) == len(("N", "n_p", "d_dim"))
    on_dev = patch_descs.is_cuda
    dev = _lib.require_cuda(patch_descs.device if on_dev else None)
    x = _as_device_f32(patch_descs, dev)
    B, N, D = x.shape
    out = torch.empty(B, D, device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().anyloc_pool(_lib.ptr(x), None, B, N, D, _POOL[method], float(gem_p),
                                           int(bool(gem_use_abs)), _lib.ptr(out), _lib.stream_ptr()), "anyloc_pool")
    return out if on_dev else out.cpu()


# ------------------------------------------------------------------ retrieval
TOPK_KERNEL_DESCRIPTION = ("retrieval: gemm_tc3_2cta_kernel<true, BIAS, hi-only> (tcgen05 cta_group::2, ONE fp16 pass = coarse "
                           "scores with a rigorous per-query error bound) over a prepared database index -> "
                           "topk_candidates_kernel -> topk_rescore_kernel (exact fp32 re-scoring of the candidates from the "
                           "(hi,lo) pairs + k-best); 3-term GEMM + topk_select2_kernel as the device-gated fallback")


class FlatIndex:
    """GPU stand-in for `faiss.IndexFlatIP` / `IndexFlatL2` as get_top_k_recall drives them (utilities.py:439-450):
    `add(db)` normalises the rows (when `norm_descs`) and stores them once as the operand pairs of the score GEMM
    (anyloc_index_add); `search(qu, k)` is exact -- k best per query, best first, lowest database index first among
    equal scores.  Rows may be added in chunks (e.g. descriptor batches as they leave the all-gather)."""

    def __init__(self, d: int, method: str = "cosine", norm_descs: bool = True, capacity: int = 0, device=None):
        if method not in _lib.METRIC:
            raise NotImplementedError(f"Method: {method}")
        self.d, self.method, self.norm_descs = int(d), method, bool(norm_descs)
        self.dp = self.d + (-self.d) % 4            # zero columns change neither norms nor scores
        self.ntotal, self.capacity = 0, 0
        self._blob, self._dev = None, (torch.device(device) if device is not None else None)
        if capacity:
            self._reserve(int(capacity), _lib.require_cuda(self._dev))

    def _reserve(self, capacity, dev):
        lib = _lib.load()
        norm = int(self.norm_descs)
        blob = torch.empty(lib.anyloc_index_bytes(capacity, self.dp, norm), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.anyloc_index_init(_lib.ptr(blob), blob.numel(), capacity, self.dp, norm, _lib.stream_ptr()),
                       "anyloc_index_init")
            if self.ntotal:         # growth: the used rows of every section move into the larger blob
                _lib.check(lib.anyloc_index_copy(_lib.ptr(blob), blob.numel(), capacity, _lib.ptr(self._blob),
                                                 self._blob.numel(), self.capacity, self.ntotal, self.dp, norm,
                                                 _lib.stream_ptr()), "anyloc_index_copy")
        self._blob, self.capacity, self._dev = blob, capacity, dev

    def reset(self):
        """faiss `index.reset()`: forget the rows, keep the allocation."""
        if self._blob is not None and self.ntotal:
            self.ntotal = 0
            self._reserve_header_only()

    def _reserve_header_only(self):
        with torch.cuda.device(self._dev):
            _lib.check(_lib.load().anyloc_index_init(_lib.ptr(self._blob), self._blob.numel(), self.capacity, self.dp,
                                                     int(self.norm_descs), _lib.stream_ptr()), "anyloc_index_init")

    def add(self, x: Union[np.ndarray, torch.Tensor]):
        on_dev = isinstance(x, torch.Tensor) and x.is_cuda
        dev = _lib.require_cuda(x.device if on_dev else self._dev)
        n = x.shape[0]
        if x.shape[1] != self.d:
            raise ValueError(f"index dimension {self.d}, got rows of {x.shape[1]}")
        if self.ntotal + n > self.capacity:
            self._reserve(max(self.ntotal + n, 2 * self.capacity if self.ntotal else 0), dev)
        lib = _lib.load()
        # host rows are streamed in chunks of <= 1 GiB so that no second full copy of the database sits in HBM
        step = n if on_dev else max(1, (1 << 30) // (self.dp * 4))
        with torch.cuda.device(dev):
            for i in range(0, n, step):
                rows = _as_device_f32(x[i:i + step], dev)
                if self.dp != self.d:
                    rows = torch.nn.functional.pad(rows, (0, self.dp - self.d))
                _lib.check(lib.anyloc_index_add(_lib.ptr(self._blob), self._blob.numel(), self.capacity,
                                                self.ntotal + i, _lib.ptr(rows), rows.shape[0], self.dp,
                                                int(self.norm_descs), _lib.stream_ptr()), "anyloc_index_add")
        self.ntotal += n

    def add_at(self, x: torch.Tensor, row_offset: int):
        """Prepare device rows `x` into rows [row_offset, row_offset + len(x)) of the (already reserved) index -- for
        callers that receive the database out of order, e.g. chunk by chunk from an all-gather (dist.py).  `ntotal`
        becomes the highest row written; the caller must fill every row below it before searching."""
        n = x.shape[0]
        if self._blob is None or row_offset < 0 or row_offset + n > self.capacity:
            raise ValueError(f"rows [{row_offset}, {row_offset + n}) outside the reserved capacity {self.capacity}")
        rows = _as_device_f32(x, self._dev)
        if self.dp != self.d:
            rows = torch.nn.functional.pad(rows, (0, self.dp - self.d))
        with torch.cuda.device(self._dev):
            _lib.check(_lib.load().anyloc_index_add(_lib.ptr(self._blob), self._blob.numel(), self.capacity, row_offset,
                                                    _lib.ptr(rows), n, self.dp, int(self.norm_descs), _lib.stream_ptr()),
                       "anyloc_index_add")
        self.ntotal = max(self.ntotal, row_offset + n)

    def search(self, qu: Union[np.ndarray, torch.Tensor], k: int, n_q_chunk: int = 4096):
        if self.ntotal == 0:
            raise ValueError("search on an empty index")
        on_dev = isinstance(qu, torch.Tensor) and qu.is_cuda
        dev = self._dev
        q = _as_device_f32(qu, dev)
        if self.dp != self.d:
            q = torch.nn.functional.pad(q, (0, self.dp - self.d))
        lib = _lib.load()
        n_q = q.shape[0]
        dist = torch.empty(n_q, k, device=dev, dtype=torch.float32)
        idx = torch.empty(n_q, k, device=dev, dtype=torch.int64)
        with torch.cuda.device(dev):
            for i in range(0, n_q, n_q_chunk):          # bounds the [n_q, n_db] score matrix
                m = min(n_q_chunk, n_q - i)
                ws = _lib.workspaces.get(dev, lib.anyloc_index_search_workspace_bytes(self.ntotal, m, self.dp,
                                                                                     int(self.norm_descs)), "topk")
                rc = lib.anyloc_index_search(_lib.ptr(self._blob), self._blob.numel(), self.capacity, self.ntotal,
                                             _lib.ptr(q[i:i + m]), m, self.dp, k, _lib.METRIC[self.method],
                                             int(self.norm_descs), _lib.ptr(dist[i:i + m]), _lib.ptr(idx[i:i + m]),
                                             _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
                _lib.check(rc, "anyloc_index_search")
        return (dist, idx) if on_dev else (dist.cpu(), idx.cpu())


def top_k_search(db: torch.Tensor, qu: torch.Tensor, k: int, method: str = "cosine",
                 norm_descs: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
    """Exact k-nearest search on the GPU (the `faiss.IndexFlatIP/L2` `add` + `search` of get_top_k_recall,
    utilities.py:435-450).  Device tensors in, device tensors out."""
    if method not in _lib.METRIC:
        raise NotImplementedError(f"Method: {method}")
    dev = _lib.require_cuda(db.device)
    index = FlatIndex(db.shape[1], method, norm_descs, capacity=db.shape[0], device=dev)
    index.add(db)
    return index.search(qu.to(dev), k)


def get_top_k_recall(top_k: List[int], db: torch.Tensor, qu: torch.Tensor, gt_pos: np.ndarray,
                     method: str = "cosine", norm_descs: bool = True, use_gpu: bool = False,
                     use_percentage: bool = True, sub_sample_db: int = 1, sub_sample_qu: int = 1) \
        -> Tuple[np.ndarray, np.ndarray, dict]:
    """utilities.py:390-469.  `use_gpu` is accepted for signature compatibility; the search always
    runs on the GPU.  Host tensors in -> host tensors out (like faiss with torch_utils)."""
    if method not in _lib.METRIC:
        raise NotImplementedError(f"Method: {method}")
    as_numpy = type(db) == np.ndarray
    if as_numpy:
        db, qu = torch.from_numpy(db), torch.from_numpy(np.asarray(qu))
    if len(qu.shape) == 1:
        qu = qu.unsqueeze(0)
    on_dev = db.is_cuda
    dev = _lib.require_cuda(db.device if on_dev else None)
    index = FlatIndex(db.shape[1], method, norm_descs, capacity=db.shape[0], device=dev)
    index.add(db)                                   # host rows are streamed in <= 1 GiB chunks
    distances, indices = index.search(_as_device_f32(qu, dev), max(top_k))
    idx_host = indices.cpu().numpy()
    recalls = dict(zip(top_k, [0] * len(top_k)))
    for i_qu, qu_retr in enumerate(idx_host):
        correct_retr = gt_pos[i_qu * sub_sample_qu]
        for i_rec in top_k:
            if np.any(np.isin(qu_retr[:i_rec] * sub_sample_db, correct_retr)):
                recalls[i_rec] += 1
    if use_percentage:
        for k in recalls:
            recalls[k] /= len(idx_host)
    if not on_dev:
        distances, indices = distances.cpu(), indices.cpu()
    if as_numpy:
        distances, indices = distances.numpy(), indices.numpy()
    return distances, indices, recalls


seed_everything()       # import side effect of the reference module (utilities.py:1011)
