"""ctypes binding of libmerv_fusion.so (the C ABI declared in include/merv_fusion.h).

The library is the product: if it is missing this module raises ImportError-grade errors loudly —
there is no Python/torch/CPU fallback for any of the entry points.
"""

from __future__ import annotations

import ctypes as C
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

PKG = os.path.dirname(os.path.abspath(__file__))
# MERV_FUSION_LIB: another build of the SAME library (A/B labs, merv_b200/build.py MERV_BUILD_TAG); never a different implementation
LIB_PATH = os.environ.get("MERV_FUSION_LIB") or os.path.join(PKG, "libmerv_fusion.so")

MERV_F32, MERV_BF16 = 0, 1
ACT_NONE, ACT_GELU_ERF = 0, 1
MAX_ENCODERS, MAX_SEGMENTS, ROWDOT_BLOCK = 8, 4, 64
ABI_VERSION = 5

ERROR_NAMES = {-1: "MERV_E_SHAPE", -2: "MERV_E_ALIGN", -3: "MERV_E_DTYPE", -4: "MERV_E_ARCH", -5: "MERV_E_CUDA", -6: "MERV_E_ARG"}


class MervError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {message}")
        self.code = code


class PoolDesc(C.Structure):
    """merv_pool_desc"""

    _fields_ = [
        ("x", c_void_p), ("y", c_void_p), ("score_vec", c_void_p), ("score_partial", c_void_p), ("batch_index", c_void_p), ("src_batch", c_int32),
        ("F", c_int32), ("H", c_int32), ("W", c_int32), ("C", c_int32), ("T", c_int32), ("S", c_int32),
        ("x_batch_stride", c_int64), ("x_frame_stride", c_int64), ("x_token_stride", c_int64),
        ("y_batch_stride", c_int64), ("y_row_stride", c_int64),
        ("shift_f", c_int32), ("shift_h", c_int32), ("shift_w", c_int32), ("reserved_", c_int32),
    ]


class FusedDesc(C.Structure):
    """merv_fused_desc"""

    _fields_ = [
        ("num_encoders", c_int32), ("B", c_int32), ("N", c_int32), ("rows_per_video", c_int32),
        ("pool", PoolDesc * 4), ("parts", c_int32 * 4),
        ("W", c_void_p * 4), ("ldw", c_int64 * 4), ("bias", c_void_p * 4), ("c", c_void_p * 4),
        ("scores", c_void_p), ("weights", c_void_p), ("bias_mix", c_void_p), ("weights_bf16", c_void_p),
        ("out", c_void_p), ("ldo", c_int64), ("out_batch_stride", c_int64),
        ("reserved_ptr_", c_void_p), ("reserved_", c_int32 * 2),
    ]


class FusedBwdDesc(C.Structure):
    """merv_fused_bwd_desc"""

    _fields_ = [
        ("B", c_int32), ("E", c_int32), ("K", c_int32), ("embed", c_int32), ("C", c_int32 * 8),
        ("weights", c_void_p), ("dweights_out", c_void_p), ("u", c_void_p), ("gsum", c_void_p),
        ("dw_partial", c_void_p * 8), ("pbar", c_void_p * 8), ("W", c_void_p * 8), ("ldw", c_int64 * 8), ("bias", c_void_p * 8),
        ("Q", c_void_p), ("Wq", c_void_p), ("Wk", c_void_p), ("in_proj_bias", c_void_p),
        ("ds", c_void_p), ("dW", c_void_p * 8), ("lddw", c_int64 * 8), ("db", c_void_p * 8),
        ("dQ", c_void_p), ("dWq", c_void_p), ("dWk", c_void_p), ("dbias", c_void_p),
        ("workspace", c_void_p), ("workspace_floats", c_size_t),
    ]


_PP = POINTER(c_void_p)
_SIGNATURES = {
    # name: (restype, argtypes) — keep in lock-step with include/merv_fusion.h (tests/test_abi.py checks the export list)
    "merv_abi_version": (c_int, []),
    "merv_last_error": (c_char_p, []),
    "merv_device_check": (c_int, []),
    "merv_num_sms": (c_int, []),
    "merv_pool3d_score_parts": (c_int, [POINTER(PoolDesc), c_int, c_int, POINTER(c_int32)]),
    "merv_pool3d": (c_int, [POINTER(PoolDesc), c_int, c_int, c_int, c_int, c_void_p]),
    "merv_linear_bias_act": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int, c_int, c_int,
                                     c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "merv_gemm_ex": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "merv_gemv_t_workspace": (c_size_t, [c_int, c_int]),
    "merv_fusion_query_vec": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "merv_affine_score_vec": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_void_p]),
    "merv_scores_from_tokens": (c_int, [_PP, POINTER(c_int32), c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int,
                                        c_int, c_void_p]),
    "merv_scores_from_tokens_ex": (c_int, [_PP, POINTER(c_int32), c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_int, c_int,
                                           c_int, c_int, c_int, c_void_p]),
    "merv_score_consts": (c_int, [c_void_p, c_int64, c_void_p, _PP, c_void_p, c_int, c_int, c_int, c_void_p]),
    "merv_layernorm": (c_int, [_PP, POINTER(c_int64), POINTER(c_int32), c_int, c_void_p, c_void_p, c_float, c_void_p, c_int64, c_int, c_int,
                               c_void_p]),
    "merv_layernorm_backward": (c_int, [_PP, POINTER(c_int64), POINTER(c_int32), c_int, c_void_p, c_int64, c_void_p, c_float, c_void_p, c_int64,
                                        c_void_p, c_int64, c_int, c_int, c_void_p]),
    "merv_scores_from_tokens_workspace": (c_size_t, [c_int, c_int, c_int, c_int]),
    "merv_scores_from_partials": (c_int, [_PP, POINTER(c_int32), _PP, c_void_p, c_int, c_int, c_int, c_void_p]),
    "merv_softmax_weights": (c_int, [c_void_p, c_void_p, _PP, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "merv_softmax_weights_ex": (c_int, [c_void_p, c_void_p, c_void_p, _PP, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "merv_fused_linear_mix_gather": (c_int, [_PP, POINTER(c_int64), _PP, POINTER(c_int64), POINTER(c_int32), c_int, c_void_p, c_void_p,
                                             c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_int, _PP, c_int, c_void_p]),
    "merv_fused_linear_mix_multicast": (c_int, [_PP, POINTER(c_int64), _PP, POINTER(c_int64), POINTER(c_int32), c_int, c_void_p, c_void_p,
                                                c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "merv_concat_linear": (c_int, [_PP, POINTER(c_int64), c_void_p, c_int64, POINTER(c_int32), c_int, c_void_p, c_void_p, c_int64, c_int, c_int,
                                   c_void_p]),
    "merv_fused_forward": (c_int, [POINTER(FusedDesc), c_void_p]),
    "merv_scores_softmax_weights": (c_int, [_PP, POINTER(c_int32), _PP, _PP, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                            c_void_p]),
    "merv_transpose": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_int64, c_int, c_void_p]),
    "merv_cross_attention": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_float, c_int,
                                     c_void_p]),
    "merv_cross_attention_backward": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64,
                                              c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "merv_cross_attention_backward_ex_workspace": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "merv_cross_attention_backward_ex": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                                 c_int64, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p, c_size_t, c_void_p]),
    "merv_add_rows": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_void_p]),
    "merv_video_colsum": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int64, c_float, c_int, c_void_p]),
    "merv_pair_dot_chunks": (c_int, []),
    "merv_wgrad_video_parts": (c_int, [c_int, c_int]),
    "merv_wgrad_video_workspace": (c_size_t, [c_int, c_int, c_int]),
    "merv_wgrad_video": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                                 c_int, c_int, c_int, c_int, c_void_p]),
    "merv_wgrad_video_ex": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                    c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "merv_pair_dot": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p]),
    "merv_pair_dot_scale": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int64, c_int, c_void_p]),
    "merv_transpose_rowscale": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int64, c_void_p, c_int64, c_int, c_int, c_void_p]),
    "merv_fused_backward_workspace": (c_size_t, [POINTER(FusedBwdDesc)]),
    "merv_fused_backward": (c_int, [POINTER(FusedBwdDesc), c_int, c_void_p]),
    "merv_gelu": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "merv_colsum_workspace": (c_size_t, [c_int, c_int]),
    "merv_colsum": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_void_p]),
    "merv_mix_backward_workspace": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "merv_mix_backward": (c_int, [_PP, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, _PP, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "merv_mix_backward_ex_workspace": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int64]),
    "merv_mix_backward_ex": (c_int, [_PP, POINTER(c_int32), c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                                     c_void_p, c_void_p, _PP, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int,
                                     c_int, c_int, c_int, c_int, c_void_p]),
    "merv_mix_backward_strided": (c_int, [_PP, POINTER(c_int32), c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                                          c_void_p, c_void_p, c_void_p, c_void_p, _PP, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_size_t, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "merv_scalar_mix_backward_workspace": (c_size_t, [c_int, c_int, c_int]),
    "merv_scalar_mix_backward": (c_int, [_PP, c_void_p, c_void_p, c_void_p, _PP, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int, c_int,
                                         c_void_p]),
    "merv_scalar_mix_backward_strided": (c_int, [_PP, c_void_p, c_int64, c_int64, c_void_p, c_void_p, _PP, c_void_p, c_void_p, c_size_t, c_int, c_int,
                                                 c_int, c_int, c_int, c_void_p]),
    "merv_scalar_fused_backward_workspace": (c_size_t, [c_int, c_int]),
    "merv_scalar_fused_backward": (c_int, [c_void_p, c_void_p, c_void_p, _PP, _PP, _PP, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int,
                                           c_void_p]),
    "merv_softmax_mix": (c_int, [_PP, POINTER(c_int32), c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "merv_softmax_mix_ex": (c_int, [_PP, POINTER(c_int32), c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int,
                                    c_void_p]),
    "merv_fused_linear_mix": (c_int, [_PP, POINTER(c_int64), _PP, POINTER(c_int64), POINTER(c_int32), c_int, c_void_p, c_void_p,
                                      c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_int, c_void_p]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None


def load() -> C.CDLL:
    """Load libmerv_fusion.so; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python merv_b200/build.py` (needs nvcc). "
            "merv_b200 has no CPU or pure-PyTorch fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    got = lib.merv_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"{LIB_PATH} has ABI version {got}, the Python binding expects {ABI_VERSION}: rebuild")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise MervError(rc, (load().merv_last_error() or b"").decode("utf-8", "replace"))


def ptr_array(ptrs) -> "C.Array":
    return (c_void_p * len(ptrs))(*[c_void_p(p) if p else c_void_p(None) for p in ptrs])


def i32_array(vals) -> "C.Array":
    return (c_int32 * len(vals))(*vals)


def i64_array(vals) -> "C.Array":
    return (c_int64 * len(vals))(*vals)
