"""ctypes binding of the C-ABI library declared in include/egs_raster.h.

There is NO fallback: if the CUDA library cannot be built/loaded, importing a product entry
point raises.  (The oracle under oracle/ is test infrastructure and is never imported here.)
"""
from __future__ import annotations

import ctypes
import threading
from ctypes import c_char_p, c_float, c_int32, c_int64, c_void_p, POINTER

from . import build as _build

_lock = threading.Lock()
_lib = None

P = c_void_p  # every device pointer travels as void*
I32, I64, F32 = c_int32, c_int64, c_float

_SIGNATURES = {
    "egs_abi_version": (c_int32, []),
    "egs_last_error_string": (c_char_p, []),
    "egs_kernel_launch_count": (c_int64, []),
    "egs_projection_fwd": (c_int32, [I32, I32, P, P, P, P, P, I32, I32, I32, P, P, I32, I32, F32, F32, F32, F32,
                                     I32, I32, I32, P, P, P, P, P, P, P, P, P]),
    "egs_projection_bwd": (c_int32, [I32, I32, P, P, P, P, I32, I32, I32, P, P, I32, I32, F32, P, P, P, P,
                                     P, P, P, P, P, P, P]),
    "egs_projection_fwd_antialiased": (c_int32, [I32, I32, P, P, P, P, P, I32, I32, I32, P, P, I32, I32, F32, F32, F32,
                                                 F32, I32, I32, I32, P, P, P, P, P, P, P, P, P, P]),
    "egs_projection_bwd_antialiased": (c_int32, [I32, I32, P, P, P, P, P, I32, I32, I32, P, P, I32, I32, F32, P, P, P,
                                                 P, P, P, P, P, P, P, P]),
    "egs_projection_fwd_raw": (c_int32, [I32, I32, P, P, P, P, P, P, I32, P, P, I32, I32, F32, F32, F32, F32,
                                         I32, I32, I32, P, P, P, P, P, P, P, P, P]),
    "egs_projection_bwd_raw": (c_int32, [I32, I32, P, P, P, P, P, P, I32, P, P, I32, I32, F32, P, P, P, P,
                                         P, P, P, P, P, P, P, P]),
    "egs_projection_bwd_viewmats_workspace_bytes": (c_int64, [I32, I32]),
    "egs_projection_bwd_viewmats": (c_int32, [I32, I32, P, P, P, P, P, I32, I32, I32, P, P, I32, I32, F32, P, P, P, P,
                                              P, P, P, P, P, P, I32, P, P, I64, P]),
    "egs_projection_bwd_raw_viewmats": (c_int32, [I32, I32, P, P, P, P, P, P, I32, P, P, I32, I32, F32, P, P, P, P,
                                                  P, P, P, P, P, P, P, P, P, I64, P]),
    "egs_projection_bwd_intrinsics_workspace_bytes": (c_int64, [I32, I32]),
    "egs_projection_bwd_intrinsics": (c_int32, [I32, I32, P, P, P, P, P, I32, I32, I32, P, P, I32, I32, F32, P, P, P,
                                                P, P, P, P, P, P, P, I32, P, P, P, I64, P]),
    "egs_projection_bwd_raw_intrinsics": (c_int32, [I32, I32, P, P, P, P, P, P, I32, P, P, I32, I32, F32, P, P, P, P,
                                                    P, P, P, P, P, P, P, P, P, P, I64, P]),
    "egs_projection_bwd_depth": (c_int32, [I32, I32, P, P, P, P, P, I32, I32, I32, P, P, I32, I32, F32, P, P, P, P,
                                          P, P, P, P, P, P, I32, P, P, P, I64, P]),
    "egs_projection_fwd_camera_model": (c_int32, [I32, I32, I32, P, P, P, P, P, I32, I32, I32, P, P, I32, I32, F32, F32,
                                                  F32, F32, I32, I32, I32, P, P, P, P, P, P, P, P, P, P]),
    "egs_projection_bwd_camera_model": (c_int32, [I32, I32, I32, P, P, P, P, P, I32, I32, I32, P, P, I32, I32, F32, P,
                                                  P, P, P, P, P, P, P, P, P, I32, P, P, P, I64, P]),
    "egs_exclusive_scan_workspace_bytes": (c_int64, [I64]),
    "egs_exclusive_scan": (c_int32, [I64, P, P, P, P, I64, P]),
    "egs_isect_emit": (c_int32, [I32, I32, P, P, P, P, I32, I32, I32, I32, I64, P, P, P]),
    "egs_radix_sort_workspace_bytes": (c_int64, [I64, I32]),
    "egs_radix_sort_pairs_u64_u32": (c_int32, [I64, P, P, P, P, I32, P, I64, POINTER(c_int32), P]),
    "egs_radix_sort_pairs_u32_u32": (c_int32, [I64, P, P, P, P, I32, P, I64, POINTER(c_int32), P]),
    "egs_isect_scan_workspace_bytes": (c_int64, [I64]),
    "egs_isect_visible_keys": (c_int32, [I32, I32, P, P, P, P, P, P, I64, P]),
    "egs_isect_sorted_workspace_bytes": (c_int64, [I32, I32, I32, I64]),
    "egs_isect_sorted": (c_int32, [I32, I32, P, P, P, P, P, P, I32, I32, I32, I64, P, I64, P, P, P, P, P]),
    "egs_exclusive_scan_gather": (c_int32, [I64, P, P, P, P, P, I64, P]),
    "egs_isect_emit_sorted": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I64, P, P, P]),
    "egs_isect_finalize": (c_int32, [I64, P, P, P, I32, I32, I32, P, P, P]),
    "egs_isect_offset_encode": (c_int32, [I64, P, I32, I32, I32, P, P]),
    "egs_rasterize_fwd": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I32, P, P, P, P, P]),
    "egs_rasterize_fwd_count": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I32, P, P, P, P, P]),
    "egs_rasterize_bwd": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I32, P, P, P, P, P, P, P]),
    "egs_rasterize_fwd_depth": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I32, P, P, P, P, P]),
    "egs_rasterize_bwd_depth": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I32, P, P, P, P, P, P, P]),
    "egs_rasterize_checkpoint_bytes": (c_int64, [I64, I32]),
    "egs_rasterize_fwd_checkpointed": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I32, P, P, P, P, I32, I32, P, P]),
    "egs_rasterize_bwd_segmented": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I32, P, P, P, P, P, P, I32, I32, P, P, P]),
    "egs_rasterize_fwd_features": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I32, I32, P, I32, I32, I32, I32,
                                             P, P, P, P, P]),
    "egs_rasterize_bwd_features": (c_int32, [I32, I32, I64, P, P, P, P, I32, I32, I32, I32, I32, P, I32, I32, I32, I32,
                                             P, P, P, P, P, P, P, P]),
    "egs_densify_stats_update": (c_int32, [I32, I32, P, P, F32, P, P, P, P]),
    "egs_l1_ssim_fwd": (c_int32, [I32, I32, I32, P, P, P, P, P, P]),
    "egs_l1_ssim_bwd": (c_int32, [I32, I32, I32, P, P, P, P, F32, P, P, P]),
    "egs_allreduce_f32_peer": (c_int32, [I32, I32, P, I64, I64, P]),
    "egs_allreduce_f32_multimem": (c_int32, [I32, I32, P, I64, I64, P]),
    "egs_fused_adam": (c_int32, [I32, P, P, P, P, P, P, F32, F32, F32, I64, P]),
    "egs_probe_fp32_fma": (c_int32, [I32, I32, P, POINTER(ctypes.c_double), P]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def load() -> ctypes.CDLL:
    """Load (building first if the in-tree library is missing or stale).  Raises on failure."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.build()  # no-op when up to date; raises RuntimeError when nvcc fails
        lib = ctypes.CDLL(str(path))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError = missing export: fail loudly
            fn.restype = res
            fn.argtypes = args
        if lib.egs_abi_version() != 1:
            raise RuntimeError(f"libegs_raster ABI {lib.egs_abi_version()} != 1 expected by the Python side")
        _lib = lib
        return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().egs_last_error_string()
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode(errors='replace') if msg else ''}")
