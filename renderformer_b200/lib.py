"""ctypes binding of the C-ABI kernel library (include/rfb200.h -> librfb200.so).

There is no CPU fallback: if the shared library is missing or a kernel returns an error the
call raises.  Tensors are passed as raw device pointers (`tensor.data_ptr()`); torch is only
used by callers for memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librfb200.so")

F32, BF16, F16 = 0, 1, 2
A_LINEAR, A_CONV3X3 = 0, 1
EPI_STORE, EPI_SWIGLU, EPI_FINAL, EPI_FINAL_RAW = 0, 1, 2, 3

_ERRORS = {-1: "bad argument / unsupported shape", -2: "misaligned pointer or stride",
           -3: "CUDA driver entry point unavailable", -4: "tensor map rejected", -5: "kernel launch failed"}


class RfbError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("A", C.c_void_p), ("lda", C.c_longlong),
        ("W", C.c_void_p), ("ldw", C.c_longlong),
        ("dtype", C.c_int), ("a_mode", C.c_int),
        ("B", C.c_int), ("H", C.c_int), ("Wd", C.c_int), ("Cin", C.c_int),
        ("epi", C.c_int),
        ("bias", C.c_void_p), ("res1", C.c_void_p), ("res2", C.c_void_p),
        ("res_dtype", C.c_int), ("ldres", C.c_longlong),
        ("out", C.c_void_p), ("out_dtype", C.c_int), ("ldo", C.c_longlong),
        ("out_act", C.c_void_p), ("row_map", C.c_void_p),
        ("w2", C.c_void_p), ("b2", C.c_void_p),
        ("bn_override", C.c_int), ("max_ctas", C.c_int),
        ("in_sumsq", C.c_void_p), ("in_sumsq_ld", C.c_int), ("in_sumsq_parts", C.c_int),
        ("in_rscale", C.c_void_p), ("scale_dim", C.c_int), ("norm_dim", C.c_int), ("norm_eps", C.c_float),
        ("out_rscale", C.c_void_p), ("out_sumsq", C.c_void_p), ("out_sumsq_ld", C.c_int),
        ("out16", C.c_void_p), ("out16_dtype", C.c_int), ("ld16", C.c_longlong),
        ("col_mul", C.c_void_p), ("aux_row_map", C.c_void_p),
        ("vt_out", C.c_void_p), ("vt_dtype", C.c_int), ("vt_split", C.c_int), ("vt_rows_per_batch", C.c_int),
        ("vt_ld", C.c_longlong), ("vt_batch_stride", C.c_longlong),
        ("crop_h", C.c_int), ("crop_w", C.c_int), ("crop_top", C.c_int), ("crop_left", C.c_int),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int), ("H", C.c_int), ("Nq", C.c_int), ("Nk", C.c_int),
        ("Q", C.c_void_p), ("ldq", C.c_longlong), ("q_batch_stride", C.c_longlong),
        ("K", C.c_void_p), ("ldk", C.c_longlong), ("k_batch_stride", C.c_longlong),
        ("Vt", C.c_void_p), ("ldvt", C.c_longlong), ("vt_batch_stride", C.c_longlong),
        ("O", C.c_void_p), ("ldo", C.c_longlong), ("o_batch_stride", C.c_longlong),
        ("key_mask_bits", C.c_void_p), ("mask_batch_stride_words", C.c_longlong),
        ("mode", C.c_int), ("group_id", C.c_void_p), ("group_period", C.c_int),
        ("scale", C.c_float),
        ("q_sumsq", C.c_void_p), ("k_sumsq", C.c_void_p), ("sumsq_ld", C.c_int), ("sumsq_parts", C.c_int),
        ("norm_dim", C.c_int),
        ("norm_eps", C.c_float),
        ("dtype", C.c_int),
        ("kv_split_tiles", C.c_int), ("split_ws", C.c_void_p), ("split_ws_bytes", C.c_longlong),
    ]


# every symbol include/rfb200.h declares (tests/test_abi.py checks the built library exports them)
SYMBOLS = [
    "rfb_version", "rfb_launch_count", "rfb_gemm", "rfb_attention", "rfb_attention_ws_bytes", "rfb_rmsnorm", "rfb_rowstat", "rfb_qknorm_rope", "rfb_qknorm_rope_table", "rfb_qkv_post",
    "rfb_token_assemble", "rfb_texture_prep", "rfb_texture_const_prep", "rfb_vn_encode", "rfb_ray_tokens", "rfb_ray_map_tokens", "rfb_ray_map", "rfb_ray_tokens_hw",
    "rfb_ray_tokens_canvas", "rfb_ray_tokens_intrinsics", "rfb_ray_tokens_lens", "rfb_intrinsics_from_fov", "rfb_ray_map_tokens_hw", "rfb_ray_map_hw", "rfb_positions",
    "rfb_pack_mask", "rfb_cast", "rfb_transpose16", "rfb_pixel_shuffle", "rfb_im2col_s2", "rfb_upsample_bilinear", "rfb_ldr_quantize",
]

_lib = None


def load() -> C.CDLL:
    """Load librfb200.so (built in-tree by __graft_entry__.build / csrc/Makefile). Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RfbError(f"{LIB_PATH} not found: build it with `make -C {os.path.join(_HERE, 'csrc')}` "
                       "(or __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    p, i, ll, f = C.c_void_p, C.c_int, C.c_longlong, C.c_float
    lib.rfb_version.restype = i
    lib.rfb_launch_count.restype = ll
    sigs = {
        "rfb_gemm": [C.POINTER(GemmArgs), p],
        "rfb_attention": [C.POINTER(AttnArgs), p],
        "rfb_rmsnorm": [p, ll, p, p, i, ll, i, i, f, p, p],
        "rfb_rowstat": [p, p, i, ll, p, i, i, i, i, p, p],
        "rfb_qknorm_rope_table": [p, ll, p, p, i, ll, i, i, i, f, p, p, ll, p],
        "rfb_qknorm_rope": [p, ll, i, p, p, i, ll, i, i, i, f, p, p, i, p],
        "rfb_qkv_post": [p, ll, p, p, ll, C.POINTER(C.c_void_p), i, i, ll, ll, i, i, f, p, p, i, i, p],
        "rfb_token_assemble": [p, p, p, p, p, p, i, p, i, i, i, i, p],
        "rfb_texture_prep": [p, p, ll, i, i, i, p],
        "rfb_texture_const_prep": [p, p, ll, i, i, i, p],
        "rfb_ldr_quantize": [p, p, ll, i, p],
        "rfb_ray_map_tokens": [p, p, i, i, p],
        "rfb_ray_map": [p, p, p, i, i, p],
        "rfb_vn_encode": [p, p, i, i, i, p],
        "rfb_ray_tokens": [p, p, i, i, p],
        "rfb_ray_map_tokens_hw": [p, p, i, i, i, p],
        "rfb_ray_map_hw": [p, p, p, i, i, i, p],
        "rfb_ray_tokens_hw": [p, p, i, i, i, p],
        "rfb_ray_tokens_canvas": [p, p, i, i, i, i, i, i, i, p],
        "rfb_ray_tokens_intrinsics": [p, p, i, i, i, i, i, i, i, p],
        "rfb_ray_tokens_lens": [p, p, i, p, i, i, i, i, i, i, i, p],
        "rfb_intrinsics_from_fov": [p, p, i, i, i, i, p],
        "rfb_positions": [p, p, p, p, i, i, i, i, p],
        "rfb_pack_mask": [p, p, i, i, i, i, p],
        "rfb_cast": [p, p, i, ll, p],
        "rfb_transpose16": [p, ll, p, ll, i, i, p],
        "rfb_pixel_shuffle": [p, p, i, i, i, i, i, p],
        "rfb_im2col_s2": [p, p, i, i, i, i, p],
        "rfb_upsample_bilinear": [p, p, i, i, i, i, i, i, p],
    }
    for name, argtypes in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = i
    lib.rfb_attention_ws_bytes.argtypes = [i, i, i, i, i]
    lib.rfb_attention_ws_bytes.restype = ll
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RfbError(f"{what} failed: {_ERRORS.get(rc, rc)} (rc={rc})")


def launch_count() -> int:
    return int(load().rfb_launch_count())
