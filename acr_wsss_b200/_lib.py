"""ctypes binding of libacr_b200.so (the C ABI declared in include/acr_b200.h).

There is deliberately no fallback: if the shared library is missing, or a call fails, a RuntimeError is
raised.  Nothing in this package routes through `oracle/` or any CPU implementation.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_longlong, c_size_t, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ACR_B200_LIB") or os.path.join(_HERE, "libacr_b200.so")      # override: A/B builds of the same ABI (scripts/)

_lib = None

# name -> (restype, argtypes); must list every symbol declared in include/acr_b200.h
SIGNATURES = {
    "acr_abi_version": (c_int, []),
    "acr_last_error_string": (c_char_p, []),
    "acr_device_is_sm100": (c_int, []),
    "acr_attn_fwd_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                  c_void_p, c_longlong, c_void_p, c_void_p]),
    "acr_attn_bwd_bf16_workspace": (c_size_t, [c_int, c_int, c_int, c_int]),
    "acr_attn_bwd_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float,
                                  c_void_p, c_longlong, c_longlong, c_void_p, c_longlong, c_longlong, c_float, c_float, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "acr_attn_fwd_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                 c_void_p, c_longlong, c_void_p]),
    "acr_attn_bwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float,
                                 c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p]),
    "acr_layernorm_fwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p, c_int, c_void_p, c_void_p,
                                  c_void_p]),
    "acr_layernorm_bwd_workspace": (c_size_t, [c_int]),
    "acr_layernorm_bwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "acr_colsum_workspace": (c_size_t, [c_int]),
    "acr_colsum_bf16": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "acr_profile_enable": (None, [c_int]),
    "acr_profile_read": (c_int, [c_char_p, POINTER(ctypes.c_double), POINTER(c_longlong)]),
    "acr_augment_batch": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "acr_sgd_momentum_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_float, c_void_p, c_void_p]),
    "acr_gelu_fwd_bf16": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p]),
    "acr_gelu_bwd_workspace": (c_size_t, [c_int]),
    "acr_gelu_bwd_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "acr_consistency_workspace": (c_size_t, [c_int, c_int, c_int]),
    "acr_consistency_fwd_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_float,
                                        c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_longlong,
                                        c_void_p, c_size_t, c_void_p]),
    "acr_getam_row0": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                               c_void_p, c_void_p, c_void_p]),
    "acr_getam_row0_batch": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "acr_affinity_sum": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "acr_affinity_refine": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "acr_affinity_refine_tc_workspace": (c_size_t, [c_int, c_int, c_int, c_int]),
    "acr_affinity_refine_tc": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "acr_patch_cam_tc": (c_int, [c_void_p, c_longlong, c_longlong, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "acr_cam_finish": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int), c_int, c_int, c_int, c_int, c_void_p,
                               POINTER(c_longlong), c_int, c_void_p, c_longlong, c_void_p, c_size_t, c_void_p]),
    "acr_label_counts_workspace": (c_size_t, [c_int, c_int, c_int]),
    "acr_cam_label_counts": (c_int, [c_void_p, c_longlong, POINTER(c_longlong), c_int, c_void_p, c_longlong, POINTER(c_longlong),
                                     c_int, POINTER(ctypes.c_double), c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "acr_label_map_counts": (c_int, [c_void_p, c_void_p, c_longlong, POINTER(c_longlong), c_int, c_int, c_void_p, c_void_p,
                                     c_size_t, c_void_p]),
    "acr_crf_head_fwd":(c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "acr_crf_head_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "acr_bilinear_up_bwd": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "acr_pamr_workspace": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "acr_pamr_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                             POINTER(c_int), c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "acr_pamr_save_workspace": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int, c_int]),
    "acr_pamr_fwd_save": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                  POINTER(c_int), c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "acr_pamr_bwd_workspace": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "acr_pamr_bwd": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                             POINTER(c_int), c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "acr_bilateral_workspace": (c_size_t, [c_int, c_int, c_int, c_int]),
    "acr_bilateral_batch": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_float,
                                    c_void_p, c_size_t, POINTER(c_int), c_void_p]),
    "acr_dense_crf_workspace": (c_size_t, [c_int, c_int, c_int, c_int]),
    "acr_dense_crf": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_float, c_float,
                              c_float, c_float, c_void_p, c_size_t, c_void_p]),
    "bilateralfilter_batch_b200": (None, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int,
                                          c_int, c_int, c_int, c_int, c_float, c_float]),
}


def lib():
    """Load (once) and return the ctypes handle; raises if the CUDA library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C acr_wsss_b200/csrc`). There is no CPU fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            if "ACR_B200_LIB" in os.environ and not hasattr(handle, name):
                continue                # an older A/B build may lack newer entry points; calling one raises AttributeError
            fn = getattr(handle, name)  # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        if handle.acr_abi_version() != 1:
            raise RuntimeError("libacr_b200.so ABI version mismatch; rebuild")
        _lib = handle
    return _lib


def last_error():
    return lib().acr_last_error_string().decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed (rc={rc}): {last_error()}")
