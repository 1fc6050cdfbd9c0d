"""ctypes binding of libamodal_b200.so (C ABI declared in include/amodal_b200.h).

The library is the product: if it is missing or cannot be loaded this module raises -- there is no Python/torch
fallback for any compute entry point.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int32, c_int64, c_size_t, c_uint32, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# ADA_B200_LIB: load another build of the same library (bring-up builds compiled with -DADA_BRINGUP carry instrumented kernels)
LIB_PATH = os.environ.get("ADA_B200_LIB") or os.path.join(_HERE, "libamodal_b200.so")

ADA_OK, ADA_EINVAL, ADA_ENODEVICE, ADA_ECUDA, ADA_ESTATE = 0, -1, -2, -3, -4

# epilogue / activation / A-operand modes (csrc/gemm.cuh)
EPI_BF16, _EPI_UNUSED, EPI_EMBED, EPI_CONVT, EPI_TAIL, EPI_SWIGLU = range(6)
EPI_RESID_F32 = 9  # out_f32 += (acc + bias) * gamma, in place through TMA (csrc/gemm.cuh)
EPI_F16 = 10       # EPI_BF16 without activation / residuals, stored as fp16 (tap map of the fused tail)
EPI_BF16_CHLN = 11  # conv + per-pixel channel LayerNorm + ReLU (bias = conv bias, gamma / aux = LN weight / bias), N <= 256
ACT_NONE, ACT_GELU, ACT_RELU = range(3)
A_LINEAR, A_CONV3X3 = range(2)


class AdaConfig(ctypes.Structure):
    _fields_ = [
        ("embed_dim", c_int32),
        ("depth", c_int32),
        ("num_heads", c_int32),
        ("ffn_kind", c_int32),
        ("ffn_hidden", c_int32),
        ("taps", c_int32 * 4),
        ("features", c_int32),
        ("out_channels", c_int32 * 4),
        ("guide_channels", c_int32),
        ("sigmoid", c_int32),
        ("pos_grid", c_int32),
        ("interpolate_offset", c_float),
        ("input_projection", c_int32),
        ("normalize_input", c_int32),
    ]


class GemmDesc(ctypes.Structure):
    _fields_ = [
        ("A", c_void_p),
        ("Bw", c_void_p),
        ("M", c_int32),
        ("N", c_int32),
        ("K", c_int32),
        ("lda", c_int32),
        ("ldb", c_int32),
        ("a_mode", c_int32),
        ("epi", c_int32),
        ("act", c_int32),
        ("batch", c_int32),
        ("H", c_int32),
        ("W", c_int32),
        ("Cin", c_int32),
        ("bias", c_void_p),
        ("gamma", c_void_p),
        ("resid_f32", c_void_p),
        ("out_f32", c_void_p),
        ("out_bf16", c_void_p),
        ("out_relu", c_void_p),
        ("resid1", c_void_p),
        ("resid2", c_void_p),
        ("aux", c_void_p),
        ("ldo", c_int32),
        ("P", c_int32),
        ("ks", c_int32),
        ("cout", c_int32),
        ("sigmoid", c_int32),
        ("force_bn", c_int32),
        ("force_cg", c_int32),
        ("conv_stride", c_int32),
        ("conv_taps", c_int32),
    ]


# name -> (restype, argtypes); this table is also what tests use to check that every symbol of the header is exported.
SIGNATURES = {
    "ada_create": (c_int32, [POINTER(AdaConfig), POINTER(c_void_p)]),
    "ada_set_weight": (c_int32, [c_void_p, c_char_p, c_void_p, POINTER(c_int64), c_int32]),
    "ada_finalize": (c_int32, [c_void_p]),
    "ada_forward": (c_int32, [c_void_p, c_void_p, POINTER(c_void_p), POINTER(c_int32), c_int32, c_void_p, c_int32,
                              c_int32, c_int32, c_void_p]),
    "ada_workspace_bytes": (c_size_t, [c_void_p]),
    "ada_launch_count": (c_int32, [c_void_p, c_int32, c_int32, c_int32]),
    "ada_read_intermediate": (c_int32, [c_void_p, c_char_p, c_void_p, c_int64]),
    "ada_set_capture": (c_int32, [c_void_p, c_int32]),
    "ada_set_graph": (c_int32, [c_void_p, c_int32]),
    "ada_set_profile": (c_int32, [c_void_p, c_int32]),
    "ada_profile_read": (c_int32, [c_void_p, c_int32, POINTER(ctypes.c_double), POINTER(ctypes.c_double),
                                   POINTER(ctypes.c_double), POINTER(c_int32)]),
    "ada_profile_records": (c_int32, [c_void_p, c_int32, POINTER(c_int32), POINTER(ctypes.c_double)]),
    "ada_destroy": (None, [c_void_p]),
    "ada_last_error": (c_char_p, []),
    "ada_device_error": (c_int32, [POINTER(c_uint32 * 4)]),
    "ada_debug_timeline": (c_int32, [POINTER(ctypes.c_longlong), c_int32]),
    "ada_interp_pos_embed_host": (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_float, c_void_p]),
    "ada_conv_tile_shape": (c_int32, [c_int32, c_int32, c_int32, c_int32, POINTER(c_int64)]),
    "ada_op_gemm": (c_int32, [POINTER(GemmDesc), c_void_p]),
    "ada_op_layernorm": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_float,
                                   c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ada_pre_image_nearest": (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32, c_int32, c_void_p]),
    "ada_pre_mask_nearest": (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "ada_post_minmax_normalize": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ada_post_blend_seam": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "ada_pre_resize_linear_batch": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32, c_void_p]),
    "ada_pre_image_nearest_batch": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int32, c_void_p]),
    "ada_pre_mask_nearest_batch": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "ada_post_minmax_normalize_batch": (c_int32, [c_void_p, c_int32, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ada_post_blend_seam_batch": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p]),
    "ada_pre_resize_cubic_normalize_batch": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32, c_void_p]),
    "ada_post_upsample_restore_batch": (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "ada_eval_sample": (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p,
                                  c_void_p, c_void_p]),
    "ada_eval_batch": (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p]),
    "ada_eval_accumulate": (c_int32, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p]),
    "ada_op_attention": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "ada_op_channel_ln_relu": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_float, c_void_p]),
    "ada_op_upsample": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "ada_op_patch_gather": (c_int32, [c_void_p, POINTER(c_void_p), POINTER(c_int32), c_int32, c_void_p, c_int32, c_int32,
                                      c_int32, c_int32, c_void_p]),
    "ada_op_tail_gather": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                     c_int32, c_void_p]),
    "ada_op_tail_mma": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                  c_int32, c_int32, c_void_p]),
    "ada_pack_tail_mma": (c_int32, [c_void_p, c_int32, c_void_p]),
    "ada_pack_tail_taps": (c_int32, [c_void_p, c_int32, c_void_p]),
    "ada_pack_conv3x3": (c_int32, [c_void_p, c_int32, c_int32, c_void_p]),
    "ada_pack_convT": (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_void_p]),
}

_lib = None


class AdaError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libamodal_b200 error {code}: {msg}")
        self.code = code


def load() -> ctypes.CDLL:
    """dlopen the CUDA library (built in-tree by __graft_entry__.build()). Raises if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no fallback implementation."
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(code: int) -> None:
    if code != ADA_OK:
        raise AdaError(code, load().ada_last_error().decode("utf-8", "replace"))


def device_error():
    arr = (c_uint32 * 4)()
    load().ada_device_error(ctypes.byref(arr))
    return list(arr)
