"""ctypes binding of libfacet_b200.so (the C ABI declared in include/facet_b200.h).

There is no CPU fallback: if the library is missing it is built with nvcc; if that fails,
or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfacet_b200.so")

_lock = threading.Lock()
_lib = None

c_u8p = C.c_void_p   # raw device/host addresses are passed as integers
_P = C.c_void_p

_SIGNATURES = {
    "fb_abi_version": (C.c_int, []),
    "fb_last_error": (C.c_char_p, []),
    "fb_launch_count": (C.c_uint64, []),
    "fb_device_sm_count": (C.c_int, []),
    "fb_profile_enable": (None, [C.c_int]),
    "fb_profile_read": (C.c_int, [_P, _P, C.c_int]),
    "fb_tech_stats": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, _P, _P, _P, C.c_int, _P]),
    "fb_tech_stats_luma": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, _P, _P, _P, C.c_int, _P, _P]),
    "fb_tech_stats_fused": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, _P, _P, _P, _P, _P, _P, _P]),
    "fb_tech_derive": (C.c_int, [_P, C.c_int, _P, _P]),
    "fb_tech_stats_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "fb_gray_hsv": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "fb_gray_plane": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "fb_canny_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "fb_canny": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_size_t, _P, _P, _P]),
    "fb_roi_laplacian": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, _P]),
    "fb_clip_preprocess": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int,
                                     _P, _P, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, C.c_int, C.c_int,
                                     _P, _P, _P, _P, _P, C.c_int, C.c_int, _P, _P]),
    "fb_phash": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, _P, _P, C.c_int, _P, _P, C.c_int,
                           _P, _P, _P, _P, _P, C.c_int, _P, C.c_int, C.c_int, _P, _P]),
    "fb_orient": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, _P, C.c_int64, _P]),
    "fb_thumbnail": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, _P,
                               _P, _P, C.c_int, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "fb_thumbnail_from_reduced": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, _P, _P,
                                            C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "fb_jpeg_encode_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "fb_jpeg_encode_out_stride": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "fb_jpeg_encode": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int64, _P, _P, C.c_int, _P, C.c_size_t, _P, C.c_int64, _P, _P]),
    "fb_jpeg_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64]),
    "fb_jpeg_decode": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, C.c_int, C.c_int64, C.c_int,
                                 _P, C.c_size_t, _P, C.c_int64, _P, _P]),
    "fb_hamming_pairs": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int, C.c_int, _P, C.c_int64, _P, _P]),
    "fb_burst_links": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int, C.c_int64, C.c_double, _P, _P, C.c_int64, _P, _P]),
}


class VitLayer(C.Structure):
    _fields_ = [(n, _P) for n in ("ln1_g", "ln1_b", "ln2_g", "ln2_b", "w_qkv", "b_qkv", "w_out", "b_out",
                                  "w_fc", "b_fc", "w_proj", "b_proj", "w_qkv_ln", "s_qkv", "c_qkv", "w_fc_ln", "s_fc", "c_fc")]


class VitWeights(C.Structure):
    _fields_ = [(n, _P) for n in ("w_patch", "class_emb", "pos_emb", "ln_pre_g", "ln_pre_b", "ln_post_g", "ln_post_b",
                                  "proj", "head_w1", "head_b1", "head_w2", "head_b2", "tag_emb")] + [
        ("n_tags", C.c_int), ("f16", C.c_int), ("n_layers", C.c_int), ("layers", C.POINTER(VitLayer)), ("fused_ln", C.c_int)]


_SIGNATURES.update({
    "fb_gemm_bf16": (C.c_int, [_P, C.c_int64, _P, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int64,
                               _P, C.c_int64, _P]),
    "fb_f32_to_bf16": (C.c_int, [_P, _P, C.c_int64, _P]),
    "fb_cosine_pairs": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_float, C.c_float, C.c_int64, C.c_int64, _P, _P,
                                  C.c_int64, _P, _P, _P, C.c_int64, _P, _P]),
    "fb_cosine_block": (C.c_int, [_P, C.c_int64, C.c_int64, _P, C.c_int64, C.c_int64, C.c_int, C.c_float, C.c_int, _P, _P, C.c_int64, _P, _P]),
    "fb_cosine_recheck": (C.c_int, [_P, C.c_int, _P, _P, C.c_int64, C.c_float, _P, _P, C.c_int64, _P, _P]),
    "fb_vit_workspace_bytes": (C.c_size_t, [C.c_int]),
    "fb_vit_forward": (C.c_int, [C.POINTER(VitWeights), _P, C.c_int, _P, C.c_size_t, _P, _P, _P, _P, _P]),
    "fb_vit_im2col": (C.c_int, [_P, C.c_int, _P, _P]),
    "fb_vit_layernorm": (C.c_int, [_P, C.c_int64, C.c_int, _P, _P, _P, _P, _P, C.c_int64, C.c_int, _P]),
    "fb_vit_attention": (C.c_int, [_P, C.c_int, _P, _P]),
    "fb_embedding_heads": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, C.c_int, _P, _P, _P]),
    "fb_vit_attention_f16": (C.c_int, [_P, C.c_int, _P, _P]),
})


def declared_symbols():
    return sorted(_SIGNATURES)


def load(build_if_missing: bool = True):
    """Load (building first if needed) and return the ctypes handle."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = os.environ.get("FACET_B200_LIB")     # kernel-variant experiments (scripts/variant_libs.sh)
        if path:
            build_if_missing = False
        else:
            path = LIB_PATH
        if build_if_missing:
            from . import build as _build
            _build.build()
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: run `python -m facet_b200.build` (needs nvcc)")
        lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)   # AttributeError here = header/library mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        if lib.fb_abi_version() != 1:
            raise RuntimeError("libfacet_b200.so ABI version mismatch; rebuild with `python -m facet_b200.build --force`")
        _lib = lib
        return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().fb_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (rc={rc}): {msg}")


def launch_count() -> int:
    return int(load().fb_launch_count())


PROFILE_CATEGORIES = ("technical", "hs_derive", "preprocess", "im2col", "gemm", "layernorm", "attention", "vit_tail",
                      "cosine", "hamming", "other")


def profile_enable(on: bool):
    load().fb_profile_enable(1 if on else 0)


def profile_read():
    """{category: (milliseconds, launches)} recorded since profile_enable(True); synchronises the device."""
    n = len(PROFILE_CATEGORIES)
    ms = (C.c_double * n)()
    cnt = (C.c_uint64 * n)()
    check(load().fb_profile_read(C.cast(ms, C.c_void_p), C.cast(cnt, C.c_void_p), n), "fb_profile_read")
    return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(PROFILE_CATEGORIES)}


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("facet_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
