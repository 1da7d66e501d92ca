"""ctypes binding of libpai_b200.so (the C-ABI declared in include/pai_b200.h).

There is no fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import contextlib
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PAI_LIB_PATH: an alternative build of the same library (e.g. csrc/build.sh -DPAI_PROFILE_ROLES), for profiling runs
LIB_PATH = os.environ.get("PAI_LIB_PATH") or os.path.join(_HERE, "libpai_b200.so")

c_int, c_float, c_void_p, c_ll = ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_longlong

# name -> argtypes, exactly the declarations of include/pai_b200.h
SIGNATURES = {
    "pai_version": [],
    "pai_reserve_sms": [c_int],
    "pai_conv4x4_fprop": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p,
                          c_int, c_float, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "pai_convT4x4s2_fprop": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int,
                             c_float, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "pai_conv4x4_wgrad": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p,
                          c_int, c_void_p],
    "pai_convT4x4s2_wgrad": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int,
                             c_void_p],
    "pai_ssim_psnr_fwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                          c_void_p, c_void_p],
    "pai_ssim_psnr_bwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                          c_void_p, c_void_p],
    "pai_bn_stats": [c_void_p, c_ll, c_int, c_int, c_void_p, c_void_p],
    "pai_bn_finalize": [c_void_p, c_ll, c_int, c_void_p, c_void_p, c_float, c_float, c_int, c_void_p, c_void_p,
                        c_void_p, c_void_p],
    "pai_bn_apply_act": [c_void_p, c_ll, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int,
                         c_float, c_void_p],
    "pai_bn_bwd_reduce": [c_void_p, c_ll, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int,
                          c_float, c_void_p, c_void_p],
    "pai_bn_bwd_apply": [c_void_p, c_ll, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int,
                         c_float, c_void_p, c_void_p, c_void_p, c_int, c_void_p],
    "pai_act_bwd": [c_void_p, c_ll, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_float, c_void_p,
                    c_void_p, c_int, c_void_p],
    "pai_colsum": [c_void_p, c_ll, c_int, c_int, c_void_p, c_void_p],
    "pai_bn_small_fwd": [c_void_p, c_ll, c_int, c_int, c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p,
                         c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_float, c_void_p, c_int, c_void_p],
    "pai_bn_small_bwd": [c_void_p, c_ll, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_float,
                         c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p],
    "pai_smallc_conv_fprop": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                              c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_float, c_void_p],
    "pai_smallc_conv_wgrad": [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                              c_int, c_int, c_void_p, c_void_p],
    "pai_im2col4x4": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "pai_pointwise_gemm": [c_void_p, c_ll, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_float, c_void_p,
                           c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "pai_pointwise_wgrad": [c_void_p, c_ll, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p],
    "pai_col2im4x4s2": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p],
    "pai_conv3x3_fprop": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_float,
                          c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "pai_conv3x3_wgrad": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p],
    "pai_maxpool2_fwd": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p],
    "pai_maxpool2_bwd": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p],
    "pai_upsample2_fwd": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p],
    "pai_upsample2_bwd": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p],
    "pai_add_act": [c_void_p, c_int, c_void_p, c_int, c_ll, c_int, c_int, c_float, c_void_p, c_int, c_void_p],
    "pai_scale_rows_fwd": [c_void_p, c_int, c_void_p, c_ll, c_int, c_int, c_void_p, c_int, c_void_p],
    "pai_scale_rows_bwd": [c_void_p, c_int, c_void_p, c_void_p, c_int, c_ll, c_int, c_int, c_void_p, c_int, c_void_p,
                           c_void_p],
    "pai_conv_plane_to_wide": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                               c_float, c_void_p, c_int, c_void_p],
    "pai_conv_wide_to_plane": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                               c_void_p, c_void_p],
    "pai_conv_plane_wide_wgrad": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                  c_void_p],
    "pai_gconv4_3x3_fprop": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p],
    "pai_gconv4_3x3_wgrad": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "pai_subsample2": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p],
    "pai_layernorm_fwd": [c_void_p, c_ll, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p],
    "pai_layernorm_bwd": [c_void_p, c_void_p, c_ll, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                          c_void_p],
    "pai_gelu_fwd": [c_void_p, c_ll, c_void_p, c_void_p],
    "pai_gelu_bwd": [c_void_p, c_void_p, c_ll, c_void_p, c_void_p],
    "pai_attn_fwd": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "pai_attn_bwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "pai_dropout_mask": [c_void_p, c_int, c_ll, c_float, c_void_p, c_void_p],
    "pai_attn_fwd_dropout": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p],
    "pai_attn_bwd_dropout": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_float, c_void_p, c_void_p,
                             c_void_p, c_void_p],
    "pai_add_dropout_layernorm_fwd": [c_void_p, c_void_p, c_ll, c_int, c_void_p, c_int, c_float, c_void_p, c_void_p,
                                      c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "pai_layernorm_bwd_dropout": [c_void_p, c_void_p, c_ll, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "pai_gelu_dropout_fwd": [c_void_p, c_ll, c_void_p, c_int, c_float, c_void_p, c_void_p],
    "pai_gelu_dropout_bwd": [c_void_p, c_void_p, c_ll, c_void_p, c_int, c_float, c_void_p, c_void_p],
    "pai_adam_pack_conv4x4": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_float, c_float,
                              c_float, c_void_p, c_void_p, c_int, c_void_p, c_void_p],
    "pai_scale_channels": [c_void_p, c_int, c_void_p, c_int, c_ll, c_int, c_void_p, c_int, c_void_p],
    "pai_conv4x4_fprop_bnstats": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p,
                                  c_void_p, c_int, c_int, c_void_p, c_int, c_void_p],
    "pai_convT4x4s2_fprop_bnstats": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p,
                                     c_void_p, c_int, c_int, c_void_p, c_int, c_void_p],
    "pai_conv4x4_dgrad_act": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_float,
                              c_void_p, c_int, c_int, c_void_p, c_int, c_void_p],
    "pai_bn_finalize_partials": [c_void_p, c_int, c_ll, c_int, c_void_p, c_void_p, c_float, c_float, c_int, c_void_p,
                                 c_void_p, c_void_p, c_void_p],
    "pai_wgrad_finish": [c_void_p, c_ll, c_void_p, c_int, c_void_p],
    "pai_adam_prepare": [c_void_p, c_float, c_float, c_float, c_void_p, c_void_p],
    "pai_check_conv2d_f32": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int,
                             c_float, c_int, c_void_p, c_void_p],
    "pai_check_batchnorm_f32": [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float,
                                c_float, c_void_p, c_void_p],
    "pai_check_act_f32": [c_void_p, c_ll, c_int, c_float, c_void_p, c_void_p],
    "pai_check_conv2d_wgrad_f32": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float,
                                   c_int, c_void_p, c_void_p, c_void_p],
    "pai_check_batchnorm_bwd_f32": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                    c_void_p],
    "pai_check_act_bwd_f32": [c_void_p, c_void_p, c_ll, c_int, c_float, c_void_p, c_void_p],
    "pai_thin_conv4x4s2_fprop": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                 c_int, c_void_p, c_int, c_int, c_float, c_void_p],
    "pai_thin_conv4x4s2_wgrad": [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "pai_thin_convT4x4s2_plane": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p],
    "pai_conv4x4_fprop_dual": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int,
                               c_float, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p],
    "pai_to_uint8": [c_void_p, c_ll, c_void_p, c_void_p],
    "pai_afmhot_u8": [c_void_p, c_int, c_ll, c_void_p, c_void_p],
    "pai_col2im4x4s1": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "pai_resize_aa_normalize_u8": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "pai_ema_multi": [c_int, c_void_p, c_void_p, c_void_p, c_float, c_void_p],
    "pai_adam_pack_conv4x4_multi": [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_float, c_float, c_float, c_float, c_float, c_void_p, c_void_p],
    "pai_adam_multi": [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_float, c_float,
                       c_float, c_void_p, c_void_p],
}
RESTYPES = {"pai_ssim_bwd_workspace_bytes": (ctypes.c_longlong, [c_int, c_int, c_int]),
            "pai_bn_small_ok": (c_int, [c_ll, c_int, c_int])}

_lib = None
launches = 0  # number of kernels this process asked the library to launch (bench.py reports it)


def load() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with thesis-pai-reconstruction_b200/csrc/build.sh "
                "(or __graft_entry__.build()); there is no CPU or PyTorch fallback")
        lib = ctypes.CDLL(LIB_PATH)
        lib.pai_last_error.restype = ctypes.c_char_p
        lib.pai_last_error.argtypes = []
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = c_int
        for name, (res, args) in RESTYPES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = res
        _lib = lib
    return _lib


def on_device(t):
    """Context manager: make ``t``'s GPU the current device (kernels are enqueued on the *current* device's
    current stream and the library keeps per-device state), so a model on cuda:1 works after cuda:0 was used."""
    import torch
    return torch.cuda.device(t.device) if t.is_cuda else contextlib.nullcontext()


def call(name: str, *args, kernels: int = 1) -> None:
    global launches
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {lib.pai_last_error().decode()}")
    launches += kernels
