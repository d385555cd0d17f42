"""ctypes binding of libattngan_b200.so (the C ABI declared in include/attngan_b200.h).

There is no CPU or PyTorch fallback: if the shared library is missing this module raises, and the
entry points themselves fail with a cudaError_t when no CUDA device is present.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_size_t, c_void_p, c_char_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libattngan_b200.so")

AGB_F32, AGB_BF16, AGB_F16 = 0, 1, 2
AGB_MATH_FP32, AGB_MATH_TC_F16, AGB_MATH_TC_BF16, AGB_MATH_TC_F16X2 = 0, 1, 2, 3
AGB_MATH_SAVE = 0x100   # flag for agb_damsm_fwd: training forward (see include/attngan_b200.h)
MATH_NAMES = {"fp32": AGB_MATH_FP32, "f16": AGB_MATH_TC_F16, "bf16": AGB_MATH_TC_BF16, "f16x2": AGB_MATH_TC_F16X2}

# name -> (restype, argtypes); mirrors include/attngan_b200.h one to one
SIGNATURES = {
    "agb_version": (c_int, []),
    "agb_last_error": (c_char_p, []),
    "agb_has_tcgen05": (c_int, []),
    "agb_tc_selftest": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "agb_tc_gemm_test": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                 c_void_p]),
    "agb_set_option": (c_int, [c_char_p, ctypes.c_longlong]),
    "agb_launch_count": (ctypes.c_longlong, []),
    "agb_prof_enable": (None, [c_int]),
    "agb_prof_read": (c_int, [c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_longlong)]),
    "agb_word_attn_fwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                                  c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                  c_int, c_int, c_int, c_void_p]),
    "agb_word_attn_bwd_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "agb_word_attn_bwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_size_t, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                  c_void_p]),
    "agb_word_attn_fwd_nhwc": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                                       c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                       c_int, c_int, c_int, c_void_p]),
    "agb_word_attn_bwd_nhwc": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_size_t, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                       c_void_p]),
    "agb_damsm_supported": (c_int, [c_int, c_int, c_int, c_int]),
    "agb_damsm_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "agb_damsm_fwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int,
                              c_int, c_int, c_int, c_float, c_float, c_float, c_int, c_void_p,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int,
                              c_void_p]),
    "agb_damsm_bwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int,
                              c_int, c_int, c_int, c_float, c_float, c_float, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_void_p]),
    "agb_damsm_cand_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "agb_damsm_cand_fwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_void_p, c_int,
                                   c_int, c_int, c_int, c_int, c_float, c_float, c_void_p, c_void_p, c_size_t, c_int,
                                   c_void_p]),
    "agb_damsm_pairs_workspace_bytes": (c_size_t, [c_int, c_int, ctypes.c_longlong, c_int, c_int, c_int, c_int]),
    "agb_damsm_pairs_fwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int, c_void_p,
                                    c_void_p, ctypes.c_longlong, c_int, c_int, c_int, c_float, c_float, c_void_p,
                                    c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "agb_damsm_pairs_train_workspace_bytes": (c_size_t, [c_int, c_int, ctypes.c_longlong, c_int, c_int, c_int,
                                                         c_int]),
    "agb_damsm_pairs_train_fwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int,
                                          c_void_p, c_void_p, ctypes.c_longlong, c_int, c_int, c_int, c_float, c_float,
                                          c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "agb_damsm_pairs_bwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int, c_void_p,
                                    c_void_p, ctypes.c_longlong, c_int, c_int, c_int, c_float, c_float, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "agb_sent_cos_pairs_bwd_workspace_bytes": (c_size_t, [c_int, c_int, ctypes.c_longlong, c_int]),
    "agb_sent_cos_pairs_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, ctypes.c_longlong, c_int,
                                       c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "agb_sent_cos_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "agb_sent_cos_pairs_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, ctypes.c_longlong, c_int,
                                       c_float, c_void_p, c_void_p]),
    "agb_sent_cos_cand_fwd": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_float, c_void_p,
                                      c_void_p]),
    "agb_sent_cos_bwd_workspace_bytes": (c_size_t, [c_int, c_int]),
    "agb_sent_cos_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "agb_contrastive_workspace_bytes": (c_size_t, [c_int]),
    "agb_contrastive_fwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_float, c_float, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "agb_region_head_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "agb_region_head_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int,
                                    c_void_p]),
    "agb_region_head_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int,
                                    c_int, c_int, c_int, c_int, c_void_p]),
    "agb_func_attention_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "agb_func_attention_fwd": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int, c_int,
                                       c_int, c_float, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                       c_void_p]),
    "agb_func_attention_bwd": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int, c_int,
                                       c_int, c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_size_t, c_void_p]),
}

_lib = None


def lib() -> ctypes.CDLL:
    """The loaded shared library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python attention-gan_b200/agb_native/build_native.py` "
                "(or __graft_entry__.build()); this package has no CPU / PyTorch fallback")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


class NativeError(RuntimeError):
    pass


def set_option(name: str, value: int) -> None:
    """process-wide tuning / test option (include/attngan_b200.h: agb_set_option)"""
    check(lib().agb_set_option(name.encode(), int(value)), f"agb_set_option({name})")


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().agb_last_error().decode("utf-8", "replace")
        kind = "invalid argument / unsupported shape" if rc < 0 else "CUDA error"
        raise NativeError(f"{what} failed with {rc} ({kind}): {msg}")
