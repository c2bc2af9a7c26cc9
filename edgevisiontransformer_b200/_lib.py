"""ctypes binding of libevt.so (the C ABI declared in include/evt.h).

There is no fallback: if the library is missing it is built with nvcc; if that fails, importing
callers get a RuntimeError.  Calls on a non-sm_100 device fail inside the library with
EVT_ERR_UNSUPPORTED -> RuntimeError.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EVT_LIB_PATH") or os.path.join(HERE, "libevt.so")   # EVT_LIB_PATH: A/B a differently built library

EVT_OK, EVT_ERR_INVALID, EVT_ERR_CUDA, EVT_ERR_UNSUPPORTED, EVT_ERR_STATE = 0, -1, -2, -3, -4
EVT_F32, EVT_BF16, EVT_TF32 = 0, 1, 2
ACT_NONE, ACT_GELU_ERF, ACT_GELU_TANH = 0, 1, 2
DIALECT_HF, DIALECT_TF = 0, 1
PREC_BF16, PREC_TF32 = 0, 1
MAX_LAYERS = 64
STAGES = ("embed", "layernorm", "qkv", "attention", "out_proj", "fc1", "fc2", "head")


class ModelSpec(C.Structure):
    _fields_ = [
        ("dialect", C.c_int), ("hidden", C.c_int), ("layers", C.c_int), ("tokens", C.c_int),
        ("image", C.c_int), ("patch", C.c_int), ("head_size", C.c_int), ("num_labels", C.c_int),
        ("act", C.c_int), ("eps", C.c_float),
        ("heads", C.c_int * MAX_LAYERS), ("inter", C.c_int * MAX_LAYERS),
        ("final_ln", C.c_int), ("head_hidden", C.c_int), ("t2t", C.c_int), ("precision", C.c_int), ("embed_k", C.c_int),
        ("head_rows", C.c_int),
    ]


class ForwardOpts(C.Structure):
    """evt_forward_opts (include/evt.h): pixel storage type, u8 normalisation, head mask, per-layer context capture."""
    _fields_ = [("pixel_dtype", C.c_int), ("pixel_scale", C.c_float * 3), ("pixel_bias", C.c_float * 3),
                ("head_mask", C.c_void_p), ("head_mask_ld", C.c_int), ("ctx_out", C.POINTER(C.c_void_p))]


PIX_F32, PIX_BF16, PIX_U8 = 0, 1, 2


SWIN_MAX_STAGES = 8


class SwinSpec(C.Structure):
    _fields_ = [("image", C.c_int), ("patch", C.c_int), ("window", C.c_int), ("embed_dim", C.c_int), ("stages", C.c_int),
                ("depths", C.c_int * SWIN_MAX_STAGES), ("heads", C.c_int * SWIN_MAX_STAGES), ("num_labels", C.c_int),
                ("eps", C.c_float), ("precision", C.c_int), ("version", C.c_int),
                ("pretrained_window", C.c_int * SWIN_MAX_STAGES), ("mask_adds", C.c_int)]


class TensorView(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ndim", C.c_int), ("shape", C.c_int64 * 4)]


_i, _i64, _f, _p, _sz = C.c_int, C.c_int64, C.c_float, C.c_void_p, C.c_size_t

# name -> (restype, argtypes); one entry per symbol declared in include/evt.h
SIGNATURES = {
    "evt_last_error": (C.c_char_p, []),
    "evt_version": (_i, []),
    "evt_device_check": (_i, []),
    "evt_launch_count": (_i64, []),
    "evt_launch_count_reset": (None, []),
    "evt_gemm_set_pair_mode": (None, [_i]),
    "evt_gemm_set_split_k": (None, [_i]),
    "evt_gemm_weights_static": (None, [_i]),
    "evt_layernorm_fwd": (_i, [_p, _i64, _p, _p, _p, _i, _i64, _p, _i64, _i, _f, _p]),
    "evt_layernorm2d_fwd": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _f, _p]),
    "evt_gemm_bias_act": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _i, _i, _p, _i, _i64, _i, _i, _i, _i64, _i, _i, _i, _p]),
    "evt_gemm_bias_act_tf32": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _i, _i, _p, _i64, _i, _i, _i, _i64, _i, _i, _i, _p]),
    "evt_gemm_bias_act_tf32_ex": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _i, _i, _p, _i, _i64, _i, _i, _i, _i64, _i, _i, _i, _p]),
    "evt_layernorm_gemm": (_i, [_p, _i64, _p, _p, _f, _p, _p, _i64, _p, _p, _i64, _i64, _i, _i, _i, _p]),
    "evt_gemm_residual_layernorm": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _p, _p, _f, _p, _i64, _i64, _i, _i, _p]),
    "evt_gemm_residual_layernorm_ex": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _p, _p, _f, _i, _p, _i64, _i64, _i, _i, _p]),
    "evt_attention_fwd": (_i, [_p, _i64, _p, _i64, _p, _i, _i, _i, _i, _f, _p]),
    "evt_attention_fwd_tf32": (_i, [_p, _i64, _p, _i64, _p, _i, _i, _i, _i, _f, _p]),
    "evt_attention_query_rows_fwd": (_i, [_p, _i64, _p, _i64, _p, _i, _i, _i, _i, _i, _f, _p]),
    "evt_attention_rel_bias_fwd": (_i, [_p, _i64, _p, _i64, _p, _p, _i, _i, _i, _i, _i, _i, _f, _p]),
    "evt_beit_score_bias": (_i, [_p, _i, _i, _p]),
    "evt_im2col_patch": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "evt_im2col_patch_ex": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "evt_patch_embed_workspace_bytes": (_i, [_i, _i, _i, _i, _i, C.POINTER(C.c_size_t)]),
    "evt_patch_embed_fwd": (_i, [_p, _i, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p]),
    "evt_prefix_tokens": (_i, [_p, _p, _p, _i, _i, _i, _i, _p]),
    "evt_cast_f32_bf16": (_i, [_p, _p, _i64, _p]),
    "evt_unfold_nhwc": (_i, [_p, _i, _p, _i64, _i, _i, _i, _i, _i, _i, _i, _p]),
    "evt_gather_layernorm": (_i, [_p, _p, _p, _p, _p, _i, _p, _i64, _i, _i, _i, _i, _f, _p]),
    "evt_window_attention_fwd": (_i, [_p, _i64, _p, _i64, _p, _i, _i64, _i, _i, _i, _f, _p]),
    "evt_window_attention_fwd_tf32": (_i, [_p, _i64, _p, _i64, _p, _i, _i64, _i, _i, _i, _f, _p]),
    "evt_layernorm_mean_tokens": (_i, [_p, _p, _p, _p, _i64, _i, _i, _f, _p]),
    "evt_layernorm_mean_tokens_ex": (_i, [_p, _p, _p, _p, _i, _i64, _i, _i, _f, _p]),
    "evt_layernorm_patch_mean": (_i, [_p, _p, _p, _p, _i64, _i, _i, _f, _p]),
    "evt_cosine_window_attention_fwd": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _i, _i, _i, _i, _i, _f, _p]),
    "evt_postnorm_residual": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _i, _i, _f, _p]),
    "evt_swinv2_cpb_table": (_i, [_p, _p, _p, _i, _i, _i, _p]),
    "evt_swinv2_score_bias": (_i, [_p, _i, _i, _i, _i, _f, _p]),
    "evt_model_create": (_i, [C.POINTER(ModelSpec), C.POINTER(_p)]),
    "evt_model_load_weights": (_i, [_p, C.POINTER(TensorView), _i, _p]),
    "evt_model_workspace_bytes": (_i, [_p, _i, C.POINTER(_sz)]),
    "evt_model_forward": (_i, [_p, _p, _i, _p, _p, _sz, _p]),
    "evt_model_forward_ex": (_i, [_p, _p, C.POINTER(ForwardOpts), _i, _p, _p, _sz, _p]),
    "evt_model_forward_embedded": (_i, [_p, _p, _i64, _i, _p, _p, _sz, _p]),
    "evt_unfold_ln_nhwc": (_i, [_p, _i, _p, _i64, _p, _p, _f, _i, _i, _i, _i, _i, _i, _i, _p]),
    "evt_performer_workspace_bytes": (_i, [_i, _i, C.POINTER(_sz)]),
    "evt_performer_fwd": (_i, [_p, _i64, _p, _p, _p, _p, _i, _i, _i, _i, _f, _p]),
    "evt_performer_mlp_fwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _f, _p]),
    "evt_performer_block_fwd": (_i, [_p, _i64, _p, _p, _p, _i, _i, _f, _p, _p, _p, _p, _p, _p, _p, _p, _f, _p]),
    "evt_token_transformer_workspace_bytes": (_i, [_i, _i, C.POINTER(_sz)]),
    "evt_token_transformer_block_fwd": (_i, [_p, _i64, _p, _p, _i, _i, _f, _p, _p, _p, _p, _p, _p, _p, _p, _f, _p]),
    "evt_model_launches_per_forward": (_i, [_p]),
    "evt_model_profile_begin": (_i, [_p]),
    "evt_model_profile_end": (_i, [_p, C.POINTER(_f), C.POINTER(_i)]),
    "evt_model_destroy": (_i, [_p]),
    "evt_swin_create": (_i, [C.POINTER(SwinSpec), C.POINTER(_p)]),
    "evt_swin_load_weights": (_i, [_p, C.POINTER(TensorView), _i, _p]),
    "evt_swin_workspace_bytes": (_i, [_p, _i, C.POINTER(_sz)]),
    "evt_swin_forward": (_i, [_p, _p, _i, _p, _p, _sz, _p]),
    "evt_swin_launches_per_forward": (_i, [_p]),
    "evt_swin_destroy": (_i, [_p]),
}

_lib = None
_lock = threading.Lock()


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if needed) libevt.so and attach the prototypes."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            if not build_if_missing:
                raise RuntimeError(f"{LIB_PATH} not built; run python -m edgevisiontransformer_b200.build")
            from . import build as _build
            _build.build()
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


class EvtError(RuntimeError):
    pass


def check(rc: int, what: str = "") -> None:
    if rc == EVT_OK:
        return
    msg = load().evt_last_error().decode("utf-8", "replace")
    text = f"libevt {what} failed ({rc}): {msg}"
    if rc == EVT_ERR_INVALID:
        raise ValueError(text)
    raise EvtError(text)
