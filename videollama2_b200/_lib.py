"""ctypes binding of libvl2.so (include/vl2.h).  There is NO fallback: if the library is missing the import of any
compute entry point raises, and on a box without an sm_100 GPU every compute call returns VL2_E_CUDA."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VL2_LIBVL2") or os.path.join(_HERE, "libvl2.so")   # override: A/B runs of two builds
LIB_PATH_F16 = os.environ.get("VL2_LIBVL2_F16") or os.path.join(_HERE, "libvl2_f16.so")   # same sources, fp16 storage

# Every symbol include/vl2.h declares (tests/test_abi.py checks the header against this list and the .so).
SYMBOLS = [
    "vl2_version", "vl2_storage_dtype", "vl2_last_error", "vl2_launch_count",
    "vl2_gemm_bf16", "vl2_gemm_skinny", "vl2_attention", "vl2_attention_decode", "vl2_debug_attn_trace", "vl2_debug_attn_timeline", "vl2_debug_gemm_trace", "vl2_gemm_plan",
    "vl2_decode_rope_append", "vl2_attention_decode_dyn", "vl2_gemv_bf16", "vl2_gemv_fp8", "vl2_attention_decode_workspace", "vl2_set_pdl", "vl2_l2_prefetch", "vl2_preprocess_frames", "vl2_preprocess_workspace",
    "vl2_layernorm", "vl2_rmsnorm", "vl2_row_sumsq", "vl2_row_stats",
    "vl2_patch_im2col", "vl2_clip_embed_finish",
    "vl2_dwconv3x3_ln_silu", "vl2_se_scale", "vl2_conv3d_im2col",
    "vl2_rope_inplace", "vl2_embed_splice", "vl2_tp_allreduce_stats", "vl2_patch_embed",
]

ACT_NONE, ACT_QUICK_GELU, ACT_SILU, ACT_GELU_ERF, ACT_SWIGLU, ACT_GELU_TANH = 0, 1, 2, 3, 4, 5
ACT_SIGMOID = 100  # vl2_gemm_skinny only


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("W", C.c_void_p), ("C", C.c_void_p),
        ("bias", C.c_void_p), ("residual", C.c_void_p), ("row_scale", C.c_void_p),
        ("lda", C.c_int64), ("ldw", C.c_int64), ("ldc", C.c_int64), ("ldr", C.c_int64),
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("act", C.c_int32), ("out_f32", C.c_int32), ("reserved", C.c_int32),
        ("bcast_out", C.c_void_p * 8), ("mc_out", C.c_void_p), ("n_bcast", C.c_int32), ("reserved2", C.c_int32),
        ("rms_sumsq_in", C.c_void_p), ("sumsq_out", C.c_void_p), ("rms_nparts", C.c_int32), ("reserved3", C.c_int32),
        ("rms_inv_dim", C.c_float), ("rms_eps", C.c_float),
        ("splitk_ws", C.c_void_p), ("splitk_ws_bytes", C.c_int64),
        ("ln_sum_in", C.c_void_p), ("ln_colsum", C.c_void_p), ("rowsum_out", C.c_void_p),
        ("conv_C", C.c_int32), ("conv_T", C.c_int32), ("conv_H", C.c_int32), ("conv_W", C.c_int32), ("conv_pad", C.c_int32),
        ("reserved4", C.c_int32),
        ("rope_tab", C.c_void_p), ("rope_cols", C.c_int32), ("rope_D", C.c_int32), ("rope_pos0", C.c_int32),
        ("reserved5", C.c_int32),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p),
        ("ldq", C.c_int64), ("ldk", C.c_int64), ("ldv", C.c_int64), ("ldo", C.c_int64),
        ("B", C.c_int32), ("S", C.c_int32), ("Hq", C.c_int32), ("Hkv", C.c_int32), ("D", C.c_int32),
        ("causal", C.c_int32), ("scale", C.c_float), ("reserved", C.c_int32),
    ]


class TpAllReduceArgs(C.Structure):
    _fields_ = [
        ("part", C.c_void_p * 8), ("xout", C.c_void_p * 8), ("stats", C.c_void_p * 8), ("pads", C.c_void_p * 8),
        ("part_mc", C.c_void_p), ("xout_mc", C.c_void_p), ("stats_mc", C.c_void_p),
        ("rank", C.c_int32), ("world", C.c_int32), ("S", C.c_int32), ("H", C.c_int32),
        ("epoch", C.c_uint32), ("inswitch_reduce", C.c_uint32),
    ]


class PatchEmbedArgs(C.Structure):
    _fields_ = [
        ("pixels", C.c_void_p), ("weight", C.c_void_p), ("pos", C.c_void_p), ("cls", C.c_void_p), ("gamma", C.c_void_p),
        ("beta", C.c_void_p), ("bias", C.c_void_p), ("out", C.c_void_p), ("scratch", C.c_void_p),
        ("F", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("P", C.c_int32), ("C", C.c_int32), ("Kpad", C.c_int32),
        ("eps", C.c_float), ("reserved", C.c_int32),
    ]


class Vl2Error(RuntimeError):
    pass


_libs = {}


def _variant(dtype) -> str:
    """Which build serves tensors of `dtype`: bf16 storage (libvl2.so) or fp16 storage (libvl2_f16.so)."""
    if dtype is None:
        return "bf16"
    name = str(dtype)
    if name.endswith("bfloat16") or name == "bf16":
        return "bf16"
    if name.endswith("float16") or name in ("f16", "half"):
        return "f16"
    raise TypeError(f"videollama2_b200 stores activations as bfloat16 or float16, not {dtype}")


def load(dtype=None) -> C.CDLL:
    """Load the library that stores 16-bit data as `dtype` (torch.bfloat16 - the default - or torch.float16) or raise.
    Never falls back to another implementation."""
    var = _variant(dtype)
    lib = _libs.get(var)
    if lib is not None:
        return lib
    path = LIB_PATH if var == "bf16" else LIB_PATH_F16
    if not os.path.exists(path):
        raise Vl2Error(
            f"{path} is missing: build it with `python -m videollama2_b200.build` (nvcc, sm_100a). "
            "videollama2_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(path)
    vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float
    lib.vl2_version.restype = C.c_int
    lib.vl2_last_error.restype = C.c_char_p
    lib.vl2_launch_count.restype = C.c_int64
    sigs = {
        "vl2_gemm_bf16": [C.POINTER(GemmArgs), vp],
        "vl2_gemm_skinny": [vp, i32, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp],
        "vl2_debug_attn_trace": [vp],
        "vl2_debug_attn_timeline": [vp],
        "vl2_debug_gemm_trace": [vp],
        "vl2_gemm_plan": [i32, i32, i32, i32, vp],
        "vl2_decode_rope_append": [vp, vp, i64, vp, i32, i32, i32, vp, i32, vp],
        "vl2_attention_decode_dyn": [vp, vp, vp, vp, i64, vp, i32, i32, i32, f32, vp, vp],
        "vl2_gemv_bf16": [vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, vp],
        "vl2_gemv_fp8": [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, vp],
        "vl2_attention_decode_workspace": [i32, i32, i32],
        "vl2_set_pdl": [i32],
        "vl2_l2_prefetch": [vp, C.c_size_t, vp],
        "vl2_preprocess_frames": [vp, vp],
        "vl2_preprocess_workspace": [vp],
        "vl2_attention_decode": [vp, vp, vp, vp, i64, i32, i32, i32, i32, f32, vp, vp],
        "vl2_attention": [C.POINTER(AttnArgs), vp],
        "vl2_layernorm": [vp, vp, vp, vp, vp, i64, i32, f32, i32, vp],
        "vl2_rmsnorm": [vp, vp, vp, i64, i32, f32, vp],
        "vl2_row_sumsq": [vp, vp, i64, i32, vp],
        "vl2_row_stats": [vp, vp, vp, i64, i32, vp],
        "vl2_patch_im2col": [vp, vp, i32, i32, i32, i32, i32, vp],
        "vl2_clip_embed_finish": [vp, vp, vp, vp, vp, vp, i32, i32, i32, f32, vp],
        "vl2_dwconv3x3_ln_silu": [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, vp],
        "vl2_se_scale": [vp, vp, i32, i32, i32, vp],
        "vl2_conv3d_im2col": [vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp],
        "vl2_rope_inplace": [vp, i64, i32, i32, i32, i32, i32, i32, i32, vp, i32, vp],
        "vl2_embed_splice": [vp, vp, i32, vp, i64, vp, i32, vp],
        "vl2_tp_allreduce_stats": [C.POINTER(TpAllReduceArgs), vp],
        "vl2_patch_embed": [C.POINTER(PatchEmbedArgs), vp],
    }
    for name, argtypes in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_size_t if name.endswith("_workspace") else C.c_int
    lib.vl2_storage_dtype.restype = C.c_int
    if int(lib.vl2_storage_dtype()) != (0 if var == "bf16" else 1):
        raise Vl2Error(f"{path} was built for the other storage type")
    _libs[var] = lib
    return lib


def check(rc: int, what: str, lib=None) -> None:
    if rc != 0:
        msgs = [l.vl2_last_error().decode(errors="replace") for l in ([lib] if lib is not None else _libs.values())]
        msg = " | ".join(m for m in msgs if m)
        exc = ValueError if rc in (-1, -2, -3) else (NotImplementedError if rc == -6 else Vl2Error)
        raise exc(f"{what} failed (code {rc}): {msg}")
