"""ctypes binding of libpsam_b200.so (the C ABI declared in include/psam_b200.h).

There is NO fallback: if the shared library is missing or a CUDA tensor is not supplied, the ops
raise.  PyTorch is used only for device memory and the current stream.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, byref, c_float, c_int, c_longlong, c_size_t, c_void_p

import torch

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG, "lib", "libpsam_b200.so")
_lib = None

ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2


class Operand(Structure):
    _fields_ = [("hi", c_void_p), ("plane_stride", c_longlong), ("rows", c_int), ("k", c_int),
                ("row_stride", c_longlong), ("nb1", c_int), ("nb2", c_int),
                ("b1_stride", c_longlong), ("b2_stride", c_longlong)]


class GemmOut(Structure):
    _fields_ = [("out_f32", c_void_p), ("ldo", c_longlong), ("out_b1", c_longlong), ("out_b2", c_longlong),
                ("out_hi", c_void_p), ("out_plane", c_longlong), ("ldo_s", c_longlong),
                ("outs_b1", c_longlong), ("outs_b2", c_longlong),
                ("bias", c_void_p), ("resid", c_void_p), ("alpha", c_float), ("act", c_int), ("accumulate", c_int),
                ("swiglu", c_int), ("tile_hint", c_int), ("gmax", c_void_p), ("ld_gmax", c_longlong), ("group_rows", c_int),
                ("rd_w", c_void_p), ("rd_out", c_void_p), ("rd_rows", c_int), ("rd_c", c_int),
                ("stats_out", c_void_p), ("ln_stats", c_void_p), ("ln_c", c_void_p), ("ln_h", c_int), ("ln_eps", c_float),
                ("variant", c_int)]


class LinearArgs(Structure):
    _fields_ = [("x", c_void_p), ("ldx", c_longlong), ("x_z", c_longlong),
                ("x2", c_void_p), ("x2_z", c_longlong),
                ("w", c_void_p), ("ldw", c_longlong), ("w_z", c_longlong),
                ("b", c_void_p), ("b_z", c_longlong),
                ("r", c_void_p), ("r_z", c_longlong),
                ("y", c_void_p), ("ldy", c_longlong), ("y_z", c_longlong),
                ("M", c_int), ("N", c_int), ("K", c_int), ("Z", c_int), ("act", c_int)]


class LnArgs(Structure):
    _fields_ = [("x", c_void_p), ("ldx", c_longlong), ("r", c_void_p), ("ldr", c_longlong),
                ("gbias", c_void_p), ("ld_gbias", c_longlong), ("group_rows", c_int),
                ("gamma", c_void_p), ("beta", c_void_p), ("eps", c_float),
                ("rows", c_int), ("D", c_int), ("act", c_int),
                ("y", c_void_p), ("ldy", c_longlong),
                ("y_hi", c_void_p), ("y_plane", c_longlong), ("ldy_s", c_longlong), ("pitch", c_longlong), ("padded", c_int), ("policy", c_int),
                ("post_add", c_void_p), ("ld_post", c_longlong), ("y2_hi", c_void_p), ("y2_plane", c_longlong), ("ldy2_s", c_longlong)]


EXPORTS = [
    "psam_fps_workspace_bytes", "psam_fps_f32", "psam_knn_f32", "psam_group_gather_f32", "psam_knn3_interp_f32", "psam_nn_distance_f32",
    "psam_voronoi_features_f32", "psam_scatter_amax_f32",
    "psam_border_prompt_workspace_bytes", "psam_border_prompt_f32",
    "psam_gemm_bf16x3", "psam_gemm_rowln_bf16x3", "psam_attention_bf16x3", "psam_attention_bf16x3_twopass", "psam_linear_f32", "psam_layernorm_f32", "psam_swiglu_ln", "psam_small_in_linear",
    "psam_group_max", "psam_softmax_split", "psam_transpose_split", "psam_posenc_f32", "psam_attention_f32",
    "psam_decoder_prepare", "psam_interp_ln_gelu", "psam_mask_dot", "psam_add_bcast_f32", "psam_split_f32", "psam_split_add_f32",
    "psam_mask_stats_f32", "psam_mask_iou_u32", "psam_mask_nms_workspace_bytes", "psam_mask_nms", "psam_mask_unpack_u8",
    "psam_version",
]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"psam_b200: native library {LIB_PATH} is missing - run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or PyTorch fallback for this path)")
        L = ctypes.CDLL(LIB_PATH)
        ll, i, f, p = c_longlong, c_int, c_float, c_void_p
        L.psam_fps_workspace_bytes.restype = c_size_t
        L.psam_fps_workspace_bytes.argtypes = [i, i, i]
        L.psam_version.restype = ctypes.c_char_p
        L.psam_border_prompt_workspace_bytes.restype = c_size_t
        L.psam_border_prompt_workspace_bytes.argtypes = [i, i, i]
        L.psam_mask_nms_workspace_bytes.restype = c_size_t
        L.psam_mask_nms_workspace_bytes.argtypes = [i, i]
        sig = {
            "psam_fps_f32": [p, i, i, i, p, p, p, p],
            "psam_knn_f32": [p, p, i, i, i, i, p, p, p],
            "psam_group_gather_f32": [p, p, p, p, p, i, i, i, i, i, i, f, p, p],
            "psam_voronoi_features_f32": [p, p, p, p, i, i, i, i, i, p, p, ll, ll, p],
            "psam_scatter_amax_f32": [p, p, i, i, i, i, p, p],
            "psam_knn3_interp_f32": [p, p, i, i, i, p, p, p],
            "psam_nn_distance_f32": [p, p, i, i, p, p, p],
            "psam_border_prompt_f32": [p, p, p, p, i, i, i, i, p, p, p, p, p],
            "psam_gemm_bf16x3": [POINTER(Operand), POINTER(Operand), POINTER(GemmOut), i, i, p],
            "psam_gemm_rowln_bf16x3": [POINTER(Operand), POINTER(Operand), p, ll, i, p, p, f, i, p, ll, ll, i, p],
            "psam_attention_bf16x3": [POINTER(Operand), POINTER(Operand), POINTER(Operand), p, ll, ll, ll, ll, f, p],
            "psam_attention_bf16x3_twopass": [POINTER(Operand), POINTER(Operand), POINTER(Operand), p, ll, ll, ll, ll, f, p],
            "psam_linear_f32": [POINTER(LinearArgs), p],
            "psam_layernorm_f32": [POINTER(LnArgs), p],
            "psam_swiglu_ln": [p, ll, ll, i, i, p, p, f, p, ll, ll, ll, p],
            "psam_small_in_linear": [p, i, i, p, p, p, p, f, i, i, i, p, ll, ll, p],
            "psam_group_max": [p, ll, i, i, i, p, ll, p, ll, ll, p],
            "psam_softmax_split": [p, ll, ll, i, f, p, ll, ll, p],
            "psam_transpose_split": [p, ll, ll, ll, ll, p, ll, ll, ll, ll, i, i, i, i, p],
            "psam_posenc_f32": [p, ll, p, i, p, p, p, p, p, p],
            "psam_attention_f32": [p, p, p, p, i, i, i, i, i, ll, ll, ll, ll, p],
            "psam_decoder_prepare": [p, p, i, p, i, p, p, ll, ll, i, i, i, i, p, p, p],
            "psam_interp_ln_gelu": [p, i, i, i, i, p, p, i, p, p, f, p, ll, ll, p],
            "psam_mask_dot": [p, ll, p, i, i, i, i, p, p],
            "psam_add_bcast_f32": [p, p, ll, ll, ll, ll, p, p],
            "psam_split_f32": [p, ll, ll, i, p, ll, ll, ll, p],
            "psam_split_add_f32": [p, p, ll, ll, i, p, ll, ll, ll, p],
            "psam_mask_stats_f32": [p, p, i, i, f, f, f, f, p, p, p, p, p],
            "psam_mask_iou_u32": [p, i, p, i, i, p, p, p],
            "psam_mask_nms": [p, p, p, p, i, i, f, p, p, p, p],
            "psam_mask_unpack_u8": [p, i, p, i, i, p, p],
        }
        for name, args in sig.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = c_int
        # experiment switch behind a debug setter of the library (the library itself reads no environment variable)
        v = os.environ.get("PSAM_ATTENTION_TILES")
        if v:
            L.psam_debug_attention_tiles(int(v))
        _lib = L
    return _lib


def available() -> bool:
    return os.path.exists(LIB_PATH)


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t) -> int:
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("psam_b200: tensor must be a CUDA tensor (this path has no CPU implementation)")
    return t.data_ptr()


LAUNCHES = [0]  # kernels launched through the C ABI (each successful call is exactly one launch)


def check(rc: int, what: str):
    LAUNCHES[0] += 1
    if rc != 0:
        kind = "invalid argument" if rc == -1 else ("unsupported configuration" if rc == -2 else f"CUDA error {rc}")
        raise RuntimeError(f"psam_b200.{what} failed: {kind}")
