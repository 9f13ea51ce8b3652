"""ctypes binding of libmagnify_b200.so (the C ABI declared in include/magnify_b200.h).

There is no CPU fallback: if the library is missing this module raises, and every wrapper
raises `MagnifyB200Error` on a non-zero status.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_int, c_int64, c_void_p, POINTER

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libmagnify_b200.so")

MGB_U8, MGB_U16, MGB_F32, MGB_F64 = 0, 1, 2, 3
MGB_EINVAL, MGB_EALIGN, MGB_EUNSUPPORTED, MGB_EIO, MGB_EFORMAT = -1, -2, -3, -4, -5


class MagnifyB200Error(RuntimeError):
    def __init__(self, fn: str, code: int, text: str):
        super().__init__(f"{fn} failed with status {code}: {text}")
        self.fn, self.code = fn, code


# name -> (argtypes); every function returns int unless listed in _SPECIAL_RESTYPE.
_P = c_void_p
_I64 = c_int64
SIGNATURES = {
    "mgb_abi_version": [],
    "mgb_error_string": [c_int],
    "mgb_sm_count": [],
    "mgb_launch_count": [],
    "mgb_l2_persist": [_P, _P, _I64, ctypes.c_float],
    "mgb_set_tma_enabled": [c_int],
    "mgb_set_stitch_variant": [c_int],
    "mgb_set_gather_loader": [c_int],
    "mgb_last_gather_path": [POINTER(ctypes.c_int32)],
    "mgb_stitch": [_P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _I64, _I64, c_int, POINTER(c_int), _P],
    "mgb_flatfield_tilemax_u16": [_P, _I64, _I64, _I64, c_int, c_int, _P, _P],
    "mgb_flatfield_maxima": [_P, c_int, c_int, _I64, _P, _P, _P, _P],
    "mgb_flatfield_maxima_generic": [_P, c_int, _I64, _I64, _I64, c_int, _P, _P, _P, _P],
    "mgb_flatfield_tables": [_P, _P, c_int, _I64, _P, _P, _P, _P],
    "mgb_flatfield_stitch_u16": [_P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _I64, _I64, c_int, _P, _P, _P, _P, _P, _P],
    "mgb_flatfield_apply_generic": [_P, _P, c_int, _I64, _I64, _I64, c_int, _P, _P, _P, _P],
    "mgb_copy2d_async": [_P, _I64, _P, _I64, _I64, _I64, c_int, _P],
    "mgb_bounding_boxes": [_P, _P, _I64, c_int, _I64, _I64, _P, _P, _P],
    "mgb_roi_gather": [_P, _I64, _I64, _I64, _I64, _I64, c_int, _P, _P, _I64, c_int, _P, _P],
    "mgb_roi_gather_stats_u16": [_P, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _I64, _P, _P, _I64, c_int, _P, _P,
                                 c_int, c_int, c_int, POINTER(c_int), _P],
    "mgb_mask_count_max": [_P, _P, _I64, _I64, _P, _P],
    "mgb_roi_gather_stats_peers_u16": [_P, _I64, _I64, _I64, _I64, _I64, _P, _P, _P, _I64, _P, _P, _I64, c_int, _P,
                                       POINTER(ctypes.c_uint64), c_int, c_int, c_int, c_int, POINTER(c_int), _P],
    "mgb_roi_stats_u16": [_P, _I64, _I64, _I64, c_int, _P, _I64, _P, _P, _P, _P],
    "mgb_roi_median_u16": [_P, _I64, _I64, _I64, c_int, _P, _I64, _P, _P, _I64, _P],
    "mgb_roi_stats_f32": [_P, _I64, _I64, _I64, c_int, _P, _I64, _P, _P, _P, _P],
    "mgb_roi_median_f32": [_P, _I64, _I64, _I64, c_int, _P, _I64, _P, _P, _I64, _P],
    "mgb_chip_masks": [_P, _P, c_int, c_int, _I64, c_int, _P, _P, _P, _P],
    "mgb_disc_halfwidths": [c_int, POINTER(ctypes.c_int32)],
    "mgb_bead_labels": [_P, _I64, _I64, _I64, _P, c_int, _P, _P],
    "mgb_bead_masks": [_P, _I64, _I64, _P, _I64, c_int, _P, _P, _P, _P],
    "mgb_mask_perimeters": [_P, _I64, c_int, _P, _P],
    "mgb_to_uint8": [_P, c_int, _I64, _I64, _P, _P, _P],
    "mgb_edge_gradients_u8": [_P, _I64, _I64, _I64, _P, _P, _P, _P],
    "mgb_gradient_order_stats": [_P, _P, _I64, _I64, POINTER(c_int64), c_int, POINTER(c_int64), _P, _P],
    "mgb_canny": [_P, _P, _I64, _I64, _I64, _P, _P, _P, POINTER(c_int), _P],
    "mgb_edge_cell_lists": [_P, _I64, _I64, _I64, c_int, _P, _P, _P, _I64, POINTER(c_int64), _P],
    "mgb_sample_circles": [_P, _P, _P, _I64, _I64, _I64, c_int, _I64, ctypes.c_float, ctypes.c_float, ctypes.c_uint64,
                           _P, _P, _P, _I64, _P, POINTER(c_int64), _P, _P],
    "mgb_gradient_angles": [_P, _P, _P, _I64, _P, _P],
    "mgb_circle_perimeter": [c_int, c_int, POINTER(ctypes.c_int32), c_int, POINTER(c_int)],
    "mgb_score_circles": [_P, _I64, _I64, _I64, _P, _P, c_int, c_int, _P, _P, _P, _P, _P],
    "mgb_order_circles": [_P, _P, _I64, _P, _P],
    "mgb_filter_neighbors_device": [_P, _I64, _I64, _I64, _I64, c_int, c_int, _P, _P, POINTER(c_int), _P],
    "mgb_filter_neighbors": [POINTER(ctypes.c_int32), _I64, c_int, POINTER(ctypes.c_uint8)],
    "mgb_tiff_open": [c_char_p, POINTER(c_void_p)],
    "mgb_tiff_close": [_P],
    "mgb_tiff_page_count": [_P, POINTER(c_int64)],
    "mgb_tiff_page_info": [_P, _I64, POINTER(c_int64)],
    "mgb_tiff_description": [_P, _I64, c_char_p, _I64],
    "mgb_tiff_read_pages": [_P, POINTER(c_int64), _I64, _P, _I64, c_int],
    "mgb_tiff_write": [c_char_p, _P, _I64, _I64, _I64, c_int, c_int, c_int, c_char_p, c_int],
    "mgb_tiff_read_files": [POINTER(c_char_p), _I64, _I64, _I64, _I64, c_int, _P, _I64, c_int],
}
_SPECIAL_RESTYPE = {"mgb_error_string": c_char_p, "mgb_launch_count": c_int64}
_NO_STATUS = {"mgb_abi_version", "mgb_error_string", "mgb_sm_count", "mgb_launch_count", "mgb_set_tma_enabled", "mgb_set_stitch_variant", "mgb_set_gather_loader"}

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing. magnify_b200 has no CPU fallback: build the CUDA library with "
            "`python -m magnify_b200.build` (needs nvcc)."
        )
    import torch  # noqa: F401  (loads the CUDA runtime the library links against dynamically)

    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.argtypes = argtypes
        fn.restype = _SPECIAL_RESTYPE.get(name, c_int)
    if lib.mgb_abi_version() != 12:
        raise ImportError("libmagnify_b200.so ABI version mismatch; rebuild with `python -m magnify_b200.build --force`")
    _lib = lib
    return lib


def error_string(code: int) -> str:
    return load().mgb_error_string(code).decode()


def call(name: str, *args) -> None:
    """Call a status-returning entry point; raise MagnifyB200Error when it fails."""
    rc = getattr(load(), name)(*args)
    if rc != 0:
        raise MagnifyB200Error(name, rc, error_string(rc))


def try_call(name: str, *args) -> int:
    """Call and return the status (for probing a fast path that may answer MGB_EALIGN)."""
    return getattr(load(), name)(*args)
