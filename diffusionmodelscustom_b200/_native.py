"""ctypes binding of include/b200ddpm.h.  No torch types cross this boundary: only data_ptr() integers and sizes.

The CUDA library is the product: if it is missing or fails to load, importing this module's functions raises —
there is no eager/PyTorch/CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2D_LIB") or os.path.join(_PKG, "libb200ddpm.so")   # B2D_LIB: an instrumented build (tools/attn_trace.py)

FAMILY_R, FAMILY_D = 0, 1
INTERP_MODES = {"bicubic": 0, "bilinear": 1, "nearest": 2}

# every symbol include/b200ddpm.h declares (tests check that the library exports all of them)
SYMBOLS = ["b2d_last_error", "b2d_abi_version", "b2d_create", "b2d_destroy", "b2d_load_weights", "b2d_set_schedule",
           "b2d_set_conditioning", "b2d_forward", "b2d_sample", "b2d_sample_host", "b2d_last_launch_count", "b2d_debug_read", "b2d_profile_step",
           "b2d_op_conv2d", "b2d_op_layernorm", "b2d_op_attention", "b2d_op_attn_block", "b2d_op_attn_block_out", "b2d_op_instnorm", "b2d_op_posterior_update", "b2d_saturation_count", "b2d_debug_attn_trace", "b2d_ensemble_run",
           "b2d_op_noise_image", "b2d_op_weighted_mse", "b2d_op_eval_daily", "b2d_op_eval_pixel", "b2d_op_histogram", "b2d_encoder_forward", "b2d_decoder_forward", "b2d_op_final_layer",
           "b2d_set_timesteps", "b2d_op_ddim_update"]


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("family", "img_size", "max_batch", "c_hr", "c_out", "has_lsm", "has_topo",
                                         "cond_channels", "num_classes", "n_heads", "attn_ff", "debug_simt_conv",
                                         "interp_mode", "stem_embedding")]


class Tensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ndim", C.c_int32), ("shape", C.c_int64 * 4)]


class OpProfile(C.Structure):
    _fields_ = [("name", C.c_char * 48), ("klass", C.c_char * 24), ("flops", C.c_double), ("bytes", C.c_double),
                ("ms", C.c_double)]


class NativeError(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(f"{LIB_PATH} is missing: build it with `python -m diffusionmodelscustom_b200.build` "
                              "(there is no fallback path)")
        L = C.CDLL(LIB_PATH)
        L.b2d_last_error.restype = C.c_char_p
        L.b2d_abi_version.restype = C.c_int
        L.b2d_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
        L.b2d_destroy.argtypes = [C.c_void_p]
        L.b2d_destroy.restype = None
        L.b2d_load_weights.argtypes = [C.c_void_p, C.POINTER(Tensor), C.c_int32]
        L.b2d_set_schedule.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]
        L.b2d_set_conditioning.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                           C.c_void_p, C.c_int32, C.c_void_p]
        L.b2d_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        L.b2d_sample.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_float, C.c_int32,
                                 C.c_void_p]
        L.b2d_sample_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_float, C.c_int32]
        L.b2d_last_launch_count.argtypes = [C.c_void_p]
        L.b2d_last_launch_count.restype = C.c_int64
        L.b2d_debug_read.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.b2d_profile_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(OpProfile),
                                       C.c_int32, C.POINTER(C.c_int32)]
        L.b2d_op_conv2d.argtypes = [C.c_void_p] * 5 + [C.c_int32, C.c_void_p] + [C.c_int32] * 12 + [C.c_void_p]
        L.b2d_op_layernorm.argtypes = [C.c_void_p] * 4 + [C.c_int32, C.c_int32, C.c_void_p]
        L.b2d_op_attention.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int32] * 4 + [C.c_void_p]
        L.b2d_op_attn_block.argtypes = [C.c_void_p] * 5 + [C.c_int32] * 4 + [C.c_void_p]
        L.b2d_op_attn_block_out.argtypes = [C.c_void_p] * 7 + [C.c_int32] * 5 + [C.c_void_p]
        L.b2d_op_instnorm.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p] + \
                                     [C.c_int32] * 3 + [C.c_void_p]
        L.b2d_op_final_layer.argtypes = [C.c_void_p] * 4 + [C.c_int32] * 4 + [C.c_void_p]
        L.b2d_op_posterior_update.argtypes = [C.c_void_p] * 6 + [C.c_int32, C.c_int32, C.c_int64, C.c_uint64, C.c_uint64,
                                                                 C.c_float, C.c_void_p]
        L.b2d_set_timesteps.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_float]
        L.b2d_op_ddim_update.argtypes = [C.c_void_p] * 4 + [C.c_int32] * 3 + [C.c_float, C.c_int32, C.c_int64, C.c_uint64,
                                                              C.c_uint64, C.c_float, C.c_void_p]
        L.b2d_op_noise_image.argtypes = [C.c_void_p] * 6 + [C.c_int32, C.c_int64, C.c_uint64, C.c_uint64, C.c_float, C.c_void_p]
        L.b2d_op_weighted_mse.argtypes = [C.c_void_p] * 3 + [C.c_float, C.c_float, C.c_void_p, C.c_int64, C.c_void_p]
        L.b2d_op_eval_daily.argtypes = [C.c_void_p] * 4 + [C.c_int32, C.c_int64, C.c_void_p]
        L.b2d_op_eval_pixel.argtypes = [C.c_void_p] * 5 + [C.c_int32, C.c_int64, C.c_void_p]
        L.b2d_op_histogram.argtypes = [C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_int32, C.c_void_p, C.c_void_p]
        L.b2d_encoder_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.c_void_p]
        L.b2d_decoder_forward.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        L.b2d_saturation_count.argtypes = [C.c_int32]
        L.b2d_saturation_count.restype = C.c_uint32
        if L.b2d_abi_version() != 1:
            raise NativeError("libb200ddpm.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise NativeError(f"b200ddpm error {rc}: {lib().b2d_last_error().decode(errors='replace')}")


def ptr(t):
    """data_ptr of a torch tensor or None -> c_void_p-compatible int."""
    return None if t is None else t.data_ptr()
