"""ctypes binding of librpst.so — the C ABI declared in include/rpst.h.

There is NO fallback: if the library is missing the import of any op fails loudly with the build
command.  PyTorch is only used by callers for device memory and streams; nothing torch-typed
crosses this boundary (pointers are `tensor.data_ptr()`, the stream is `cuda_stream`)."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_void_p

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RPST_LIB") or os.path.join(PKG, "librpst.so")   # RPST_LIB: A/B a second build

RPST_OK = 0
RPST_ERR_INVALID = -1
RPST_ERR_CUDA = -2
RPST_ERR_WORKSPACE = -3
RPST_ERR_UNSUPPORTED = -4

P = c_void_p  # every device pointer and the stream travel as void*

# name -> (restype, argtypes); mirrors include/rpst.h one to one (tests/test_abi.py checks that)
SIGNATURES = {
    "rpst_version": (c_int, []),
    "rpst_last_error": (c_char_p, []),
    "rpst_set_tuning": (c_int, [c_char_p, c_int64]),
    "rpst_get_tuning": (c_int64, [c_char_p]),
    "rpst_stats_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "rpst_stats_nchw": (c_int, [P, c_int64, c_int64, c_float, P, P, P, c_size_t, P]),
    "rpst_adain_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_adain_fwd": (c_int, [P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_float, P, P, c_size_t, P]),
    "rpst_adain_fwd_mapped": (c_int, [P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_float, P, P, P, c_size_t, P]),
    "rpst_adain_bwd_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_adain_bwd": (c_int, [P, P, P, P, P, P, c_int64, c_int64, c_int64, P, c_size_t, P]),
    "rpst_plane_affine": (c_int, [P, P, P, P, c_int64, c_int64, P]),
    "rpst_pair_stats_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "rpst_pair_stats": (c_int, [P, P, c_int64, c_int64, c_float, P, P, P, c_size_t, P]),
    "rpst_plane_affine2": (c_int, [P, P, P, P, P, P, c_int64, c_int64, P]),
    "rpst_pair_loss_bwd": (c_int, [P, P, P, P, c_int, c_int, P, c_int64, c_int64, P]),
    "rpst_seg_adain_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64]),
    "rpst_pairwise_sqdist_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_pairwise_sqdist": (c_int, [P, P, c_int64, c_int64, c_int64, P, P, c_size_t, P]),
    "rpst_mrf_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int]),
    "rpst_mrf_match": (c_int, [P, P, c_int64, c_int64, c_int, c_int, c_int, P, P, P, P, c_int, P, c_size_t, P]),
    "rpst_packed_operand_bytes": (c_size_t, [c_int64, c_int64]),
    "rpst_pack_operand": (c_int, [P, c_int64, c_int64, c_int64, c_int64, P, P, P, P]),
    "rpst_gemm_packed": (c_int, [P, P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_int, c_float, P, P, P]),
    "rpst_sym_eig_fn_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "rpst_sym_eig_fn": (c_int, [P, c_int64, c_int64, c_double, P, P, P, P, P, c_size_t, P]),
    "rpst_spd_roots_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "rpst_spd_roots": (c_int, [P, c_int64, c_int64, c_double, c_double, P, P, P, P, c_size_t, P]),
    "rpst_wct_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64]),
    "rpst_wct_fuse": (c_int, [P, P, P, c_int64, c_int64, c_int64, c_int64, c_int, c_int, P, P, c_size_t, P]),
    "rpst_sanet_attn_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_sanet_attn_fwd": (c_int, [P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_int, P, P, c_size_t, P]),
    "rpst_sanet_attn_bwd_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_sanet_attn_bwd": (c_int, [P, P, P, P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_int, P, c_size_t, P]),
    "rpst_sanet_attn_clamped_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_sanet_attn_clamped_fwd": (c_int, [P, P, P, P, c_int, c_float, P, c_int64, c_int64, c_int64, c_int64, c_int, P, c_size_t, P]),
    "rpst_sanet_attn_clamped_bwd": (c_int, [P, P, P, P, c_int, c_float, P, P, P, P, P, c_int64, c_int64, c_int64, c_int64,
                                            c_int, P, c_size_t, P]),
    "rpst_cosine_affinity_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_cosine_affinity": (c_int, [P, P, P, c_int64, c_int64, c_int64, c_int64, P, c_size_t, P]),
    "rpst_sanet_adaptive_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int64]),
    "rpst_sanet_attn_adaptive_fwd": (c_int, [P, P, P, P, P, c_int64, P, P, P, P, c_int, c_float, c_float, c_float,
                                             P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_int64, c_int, P, c_size_t, P]),
    "rpst_conv1x1_stats_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_conv1x1": (c_int, [P, P, P, P, P, P, P, P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_int, c_float, c_int, P]),
    "rpst_conv1x1_stats_finalize": (c_int, [P, c_int64, c_int64, c_int64, c_float, P, P, P]),
    "rpst_sanet_attn_packed_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_sanet_attn_fwd_packed": (c_int, [P, P, P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_int, P, c_size_t, P]),
    "rpst_seg_adain_fwd": (c_int, [P, P, P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_float, P, P, c_size_t, P]),
    "rpst_seg_adain_fwd_mapped": (c_int, [P, P, P, P, P, P, c_int64, c_int64, c_int64, c_int64, c_int64, c_float,
                                          P, P, P, P, c_size_t, P]),
}


# white-box test hooks (include/rpst_debug.h): only in librpst_debug.so, never in the product library
DEBUG_LIB_PATH = os.path.join(PKG, "librpst_debug.so")
DEBUG_SIGNATURES = {
    "rpst_debug_adain_schedule": (c_int, [c_int64, c_int64, c_int, c_int, c_int, P, c_int64, P, P]),
    "rpst_debug_seg_schedule": (c_int, [c_int64, c_int64, c_int64, c_int64, c_int, P, c_int64, P, P]),
    "rpst_debug_wct_covariances_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rpst_debug_wct_covariances": (c_int, [P, c_int64, c_int64, c_int64, c_int, c_double, c_int, P, P, P, P, c_size_t, P]),
    "rpst_debug_dgemm_batched": (c_int, [P, P, P, c_int64, c_int64, P]),
    "rpst_last_error": (c_char_p, []),
    "rpst_set_tuning": (c_int, [c_char_p, c_int64]),     # the debug library keeps its own knobs
    "rpst_get_tuning": (c_int64, [c_char_p]),
}


class RpstError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"librpst error {code}: {message}")
        self.code = code


_lib = None


def lib() -> ctypes.CDLL:
    """Load librpst.so (once).  Raises if it has not been built — there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  rpst has no CPU or PyTorch fallback.")
    handle = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return handle


_debug_lib = None


def debug_lib() -> ctypes.CDLL:
    """librpst_debug.so (tests only): the product sources compiled with -DRPST_DEBUG_EXPORTS."""
    global _debug_lib
    if _debug_lib is None:
        if not os.path.exists(DEBUG_LIB_PATH):
            raise RuntimeError(f"{DEBUG_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`")
        handle = ctypes.CDLL(DEBUG_LIB_PATH)
        for name, (res, args) in DEBUG_SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _debug_lib = handle
    return _debug_lib


def check(code: int) -> None:
    if code != RPST_OK:
        msg = lib().rpst_last_error()
        raise RpstError(code, msg.decode() if msg else "")


def set_tuning(name: str, value: int) -> None:
    check(lib().rpst_set_tuning(name.encode(), int(value)))


def get_tuning(name: str) -> int:
    return int(lib().rpst_get_tuning(name.encode()))
