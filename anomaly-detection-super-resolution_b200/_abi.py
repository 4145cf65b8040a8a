"""ctypes binding of the C ABI declared in include/adsr_b200.h (libadsr_b200.so, built in-tree).

There is deliberately NO fallback: if the shared library is missing or a call returns a non-zero
status a RuntimeError is raised.  Status codes become Python exceptions here (the C side never
aborts or prints), mirroring the reference where every failure on this path is a Python exception.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
# ADSR_LIB: developer override for A/B timing of two builds in one session (tools/build_variant.sh); never a fallback
LIB_PATH = os.environ.get("ADSR_LIB") or os.path.join(_HERE, "libadsr_b200.so")
ABI_VERSION = 21

ACT_NONE, ACT_LRELU, ACT_GELU, ACT_RELU = 0, 1, 2, 3
OUT_ROWS, OUT_PIXEL_SHUFFLE2 = 0, 1

_SIGNATURES = {
    "adsr_abi_version": (c_int, []),
    "adsr_status_string": (c_char_p, [c_int]),
    "adsr_device_check": (c_int, [POINTER(c_int)]),
    "adsr_tc_gemm_bf16": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                  c_float, c_float, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_void_p, c_float,
                                  c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "adsr_swin_mlp_bf16": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int, c_float, c_void_p, c_int, c_int, c_void_p, c_int64, c_int, c_int, c_void_p]),
    "adsr_swin_mlp_adjust_bf16": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_int, c_float, c_void_p, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p, c_int64,
                                          c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "adsr_swin_mlp_conv_res_bf16": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                            c_int, c_float, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p, c_int64, c_int,
                                            c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "adsr_swin_attn_mode": (c_int, [c_int, c_int, c_int, c_int]),
    "adsr_swin_attn_bf16": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_int,
                                    c_void_p, c_int64, c_void_p, c_int, c_int, c_int, c_void_p]),
    "adsr_conv3x3_igemm_bf16": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                                        c_int, c_int, c_int, c_float, c_float, c_void_p, c_int64, c_void_p, c_int64,
                                        c_int, c_int, c_int, c_int, c_void_p]),
    "adsr_conv3x3_halo_bf16": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                                       c_float, c_void_p, c_int64, c_int, c_int, c_void_p, c_int, c_void_p]),
    "adsr_channel_mean_parts": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_int, c_void_p]),
    "adsr_layernorm_rows": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_float,
                                    c_void_p]),
    "adsr_window_attention": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                      c_int, c_int, c_int, c_void_p]),
    "adsr_window_index_map": (c_int, [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "adsr_ln_shift_partition": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_float, c_int, c_int,
                                        c_int, c_int, c_int, c_int, c_void_p]),
    "adsr_window_reverse_unshift": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int,
                                            c_int, c_void_p]),
    "adsr_drct_head": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_float, c_void_p,
                               c_void_p, c_float, c_int, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int, c_void_p]),
    "adsr_conv_last_quant": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                     c_float, c_float, c_void_p, c_void_p, c_void_p]),
    "adsr_u8_to_float_nchw": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "adsr_quantize_u8": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "adsr_score_images": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, POINTER(c_int32), c_int, c_void_p,
                                  c_void_p]),
    "adsr_anomaly_maps": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p]),
    "adsr_gms_workspace_bytes": (c_int64, [c_int, c_int, c_int]),
    "adsr_gms_map": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "adsr_localisation_workspace_bytes": (c_int64, [c_int64]),
    "adsr_localisation_metrics": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int64, c_double, c_void_p, c_int64, c_void_p,
                                          c_void_p]),
    "adsr_score_quantile": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "adsr_threshold_metrics": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int, c_float, c_void_p, c_int64, c_void_p, c_void_p]),
    "adsr_regions_workspace_bytes": (c_int64, [c_int, c_int, c_int]),
    "adsr_label_regions": (c_int, [c_void_p, c_float, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64,
                                   c_void_p]),
    "adsr_region_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                  c_void_p, c_void_p, c_int64, c_void_p]),
    "adsr_pack_slab_sw128": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p]),
    "adsr_pack_tiles_sw128": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "adsr_drct_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int]),
    "adsr_score_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int]),
    "adsr_l1_loss_grad": (c_int, [c_void_p, c_void_p, c_int64, c_float, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "adsr_conv_last_bwd_workspace_bytes": (c_int64, [c_int, c_int, c_int]),
    "adsr_conv_last_bwd": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int64, c_void_p,
                                   c_void_p, c_void_p, c_void_p]),
    "adsr_adam_step": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_float, c_float, c_float, c_int, c_void_p]),
    "adsr_validate_images": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, POINTER(c_int64), POINTER(c_int64), c_float,
                                     c_int, c_void_p, c_void_p]),
    "adsr_score_images_strided": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, POINTER(c_int64),
                                          POINTER(c_int64), c_float, c_int, c_int, c_double, c_double, c_double,
                                          POINTER(c_int32), c_int, c_void_p, c_void_p]),
    "adsr_bicubic_affine": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "adsr_conv3x3_small": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int64,
                                   c_void_p, c_int64, c_int, c_void_p]),
    "adsr_channel_mean": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_int64, c_void_p]),
    "adsr_rcab_ca_scale": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int, c_int, c_int,
                                   c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "This package has no CPU / PyTorch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)   # AttributeError if the .so does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        if handle.adsr_abi_version() != ABI_VERSION:
            raise RuntimeError("libadsr_b200.so ABI version mismatch; rebuild")
        _lib = handle
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().adsr_status_string(status).decode()
        raise RuntimeError(f"{what}: adsr status {status} ({msg})")


_num_sms = None


def num_sms() -> int:
    """SM count of the current CUDA device; raises unless it is an sm_100 part."""
    global _num_sms
    if _num_sms is None:
        n = c_int(0)
        check(lib().adsr_device_check(ctypes.byref(n)), "adsr_device_check")
        _num_sms = n.value
    return _num_sms


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
