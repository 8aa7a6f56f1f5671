"""ctypes binding of libanyloc_b200.so (C ABI in include/anyloc_b200.h).

There is no CPU fallback: if the library is missing, or no CUDA device is usable,
every compute entry point raises."""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libanyloc_b200.so")

# constants of include/anyloc_b200.h
DIST = {"cosine": 0, "euclidean": 1}
METRIC = {"cosine": 0, "l2": 1}
FACET = {"query": 0, "key": 1, "value": 2, "token": 3}
DESC = {"plain": 0, "l2": 1, "interleaved": 2}
FFN = {"mlp": 0, "swiglufused": 1}
EPI = {"bias": 0, "bias_split": 1, "gelu_split": 2, "swiglu_split": 3, "ls_resid": 4}
ENGINE = {"auto": 0, "simt": 1, "tc3": 2}
PAIR = {"tf32": 0, "f16": 1}
ACT_SCALE = 8.0     # kActScale in csrc/common.cuh


class AnylocError(RuntimeError):
    pass


class VitCfg(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("embed_dim", "depth", "num_heads", "ffn_kind", "ffn_hidden", "patch",
                                       "pair_dtype", "stride")]


_BLOCK_FIELDS = ["ln1_w", "ln1_b", "qkv_w_hi", "qkv_w_lo", "qkv_b", "proj_w_hi", "proj_w_lo", "proj_b",
                 "ls1", "ln2_w", "ln2_b", "in_w_hi", "in_w_lo", "in_b", "out_w_hi", "out_w_lo", "out_b", "ls2"]


class VitBlock(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in _BLOCK_FIELDS] + \
               [(n, C.c_float) for n in ("qkv_alpha", "proj_alpha", "in_alpha", "out_alpha")]


class VitWeightsStruct(C.Structure):
    _fields_ = [("patch_w_hi", C.c_void_p), ("patch_w_lo", C.c_void_p), ("patch_b", C.c_void_p),
                ("cls_token", C.c_void_p), ("blocks", C.POINTER(VitBlock)), ("patch_alpha", C.c_float)]


_SIGS = {
    "anyloc_last_error": (C.c_char_p, []),
    "anyloc_version": (C.c_int, []),
    "anyloc_launch_count": (C.c_longlong, []),
    "anyloc_profile_enable": (C.c_int, [C.c_int]),
    "anyloc_profile_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_double)]),
    "anyloc_device_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    "anyloc_vlad_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "anyloc_vlad_generate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 7 +
                             [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_vlad_prepared_bytes": (C.c_size_t, [C.c_int] * 2),
    "anyloc_vlad_prepare": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_vlad_generate_prepared": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t] +
                                      [C.c_int] * 7 + [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_vlad_generate_soft": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 4 + [C.c_float] +
                                  [C.c_int] * 2 + [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_preprocess_u8": (C.c_int, [C.c_void_p] + [C.c_int] * 7 + [C.POINTER(C.c_float)] * 2 +
                             [C.c_void_p, C.c_void_p]),
    "anyloc_preprocess_resize_u8": (C.c_int, [C.c_void_p] + [C.c_int] * 10 + [C.POINTER(C.c_float)] * 2 +
                                    [C.c_void_p, C.c_void_p]),
    "anyloc_pool": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 4 + [C.c_float, C.c_int, C.c_void_p, C.c_void_p]),
    "anyloc_vlad_residuals": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 4 + [C.c_void_p, C.c_void_p]),
    "anyloc_vlad_from_residuals_workspace_bytes": (C.c_size_t, [C.c_int] * 2),
    "anyloc_vlad_from_residuals": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 4 +
                                   [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_vlad_assign": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 4 +
                           [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_kmeans_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "anyloc_kmeans_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 3 +
                             [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_topk_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "anyloc_topk": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 6 +
                    [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_index_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.c_int]),
    "anyloc_index_init": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "anyloc_index_copy": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int64, C.c_void_p, C.c_size_t, C.c_int64, C.c_int64,
                                    C.c_int, C.c_int, C.c_void_p]),
    "anyloc_index_add": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int64, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p]),
    "anyloc_index_search_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.c_int, C.c_int]),
    "anyloc_index_search": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int64, C.c_int64, C.c_void_p] + [C.c_int] * 5 +
                            [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_allgather_desc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "anyloc_vit_patch_k": (C.c_int, [C.c_int]),
    "anyloc_vit_workspace_bytes": (C.c_size_t, [C.POINTER(VitCfg), C.c_int, C.c_int, C.c_int]),
    "anyloc_vit_extract": (C.c_int, [C.POINTER(VitCfg), C.POINTER(VitWeightsStruct), C.c_void_p,
                                     C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "anyloc_log_bin": (C.c_int, [C.c_void_p] + [C.c_int] * 5 + [C.c_void_p, C.c_void_p]),
    "anyloc_gemm_nt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "anyloc_split_tf32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "anyloc_split_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_void_p]),
    "anyloc_layernorm_split": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float,
                                         C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "anyloc_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                   C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "anyloc_l2_normalize_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
}
EXPORTS = sorted(_SIGS)

_lib = None


def load():
    """dlopen the library (does not need a GPU)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise AnylocError(
                f"{LIB_PATH} is missing -- build it with `python -m anyloc_b200.build` "
                "(anyloc_b200 has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def last_error():
    return load().anyloc_last_error().decode()


def check(rc, what):
    if rc != 0:
        raise AnylocError(f"{what} failed (rc={rc}): {last_error()}")


def require_cuda(device=None):
    if not torch.cuda.is_available():
        raise AnylocError("anyloc_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    load()
    dev = torch.device("cuda" if device is None else device)
    if dev.type != "cuda":
        raise AnylocError(f"anyloc_b200 runs on CUDA devices only (got device={device!r}); no CPU fallback")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    if t is None:
        return C.c_void_p(0)
    assert t.is_cuda and t.is_contiguous(), "device-contiguous tensor required"
    return C.c_void_p(t.data_ptr())


class _WorkspacePool:
    """Grow-only per-device byte buffers reused across calls (caller-owned workspaces of the C ABI)."""

    def __init__(self):
        self._bufs = {}

    def get(self, device, nbytes, tag="default"):
        key = (device.index, tag)
        buf = self._bufs.get(key)
        if buf is None or buf.numel() < nbytes:
            self._bufs.pop(key, None)
            buf = None
            buf = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
            self._bufs[key] = buf
        return buf

    def clear(self):
        self._bufs.clear()


workspaces = _WorkspacePool()

PROF_CATEGORIES = ["gemm_tc", "gemm_simt", "attention", "layernorm", "vit_misc", "vlad", "topk", "log_bin"]


def profile_enable(on=True):
    check(load().anyloc_profile_enable(int(bool(on))), "profile_enable")


def profile_read():
    """-> {category: (device_ms, launch_groups, algorithmic_work)} since the last read."""
    n = len(PROF_CATEGORIES)
    ms, groups, work = (C.c_double * n)(), (C.c_longlong * n)(), (C.c_double * n)()
    check(load().anyloc_profile_read(ms, groups, work), "profile_read")
    return {c: (ms[i], groups[i], work[i]) for i, c in enumerate(PROF_CATEGORIES)}


def launch_count():
    return int(load().anyloc_launch_count())
