"""ctypes binding of include/vi_b200.h.  There is no CPU fallback: if the
shared library is missing or a call fails, this raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _build

VI_OK = 0
VI_ERR_ARG, VI_ERR_CUDA, VI_ERR_UNSUPPORTED, VI_ERR_TOO_LARGE = -1, -2, -3, -4
STATUS_OK, STATUS_NG, STATUS_ROI_EMPTY, STATUS_SEGMENTED = 0, 1, 2, 3
MASKS_BYTES, MASKS_PACKED, MASKS_NONE = 0, 1, 2


class ViParams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("seg_method", "gaussian_blur", "morph_kernel", "adapt_block", "adapt_C",
                                         "defect_method", "threshold", "min_area", "erode_px", "median_ksize")] + \
               [("max_area_frac", C.c_double)]


class ViExcl(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("shape", "a", "b", "c", "d")]


RECORD_DTYPE = np.dtype([
    ("image", "<i4"), ("unit", "<i4"), ("otsu_t", "<i4"), ("seg_area", "<i4"), ("roi_area", "<i4"),
    ("defect_area", "<i4"), ("n_kept", "<i4"), ("status", "<i4"), ("dx", "<i4"), ("dy", "<i4"),
    ("cx", "<f8"), ("cy", "<f8"), ("n_ambiguous", "<i4"), ("n_runs", "<i4"),
])
assert RECORD_DTYPE.itemsize == 64

# vi_defect_blob: one kept defect component, unit-local (bounding box, filled-contour pixel area, 2 * contourArea, mean x / y)
BLOB_DTYPE = np.dtype([
    ("x", "<i4"), ("y", "<i4"), ("w", "<i4"), ("h", "<i4"), ("area", "<i4"), ("area2", "<i4"), ("cx", "<f8"), ("cy", "<f8"),
])
assert BLOB_DTYPE.itemsize == 40
MAX_BLOBS_PER_UNIT = 1024

EXPORTS = [
    "vi_last_error", "vi_version", "vi_params_default", "vi_ctx_create", "vi_ctx_destroy", "vi_set_grid",
    "vi_set_exclusions", "vi_set_ref_centroids", "vi_unit_pixels", "vi_unit_offsets", "vi_inspect_batch",
    "vi_inspect_batch_host", "vi_inspect_batch_host_fmt", "vi_inspect_batch_host_blobs", "vi_segment_batch", "vi_segment_batch_host", "vi_set_defect_blob_output", "vi_set_packed_mask_output", "vi_packed_mask_bytes",
    "vi_packed_mask_offsets", "vi_host_upload_bytes", "vi_peer_table_create", "vi_peer_table_open", "vi_peer_table_close",
    "vi_peer_table_destroy", "vi_peer_table_read", "vi_set_record_peers", "vi_segment_cell", "vi_fill_internal_holes", "vi_mask_stats", "vi_erode_square",
    "vi_label_components", "vi_detect_defects", "vi_ingest_argb32", "vi_ingest_gray16", "vi_set_seg_stats_output", "vi_debug_set_profile", "vi_debug_check_word", "vi_debug_fastdiv_check", "vi_debug_otsu",
    "vi_debug_rank_residual", "vi_debug_adaptive_taps",
]

_lib = None


class ViError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"vi_b200 error {code}: {msg}")
        self.code = code


def load():
    """dlopen the in-tree library (built by __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    # VI_B200_LIB=checked selects the self-checked build of the same sources (vi_debug_check_word)
    path = _build.CHECKED_LIB_PATH if os.environ.get("VI_B200_LIB") == "checked" else _build.LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the CUDA extension is the product; there is no CPU fallback)")
    lib = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    P = C.POINTER
    lib.vi_last_error.restype = C.c_char_p
    lib.vi_version.restype = C.c_int
    lib.vi_params_default.argtypes = [P(ViParams)]
    lib.vi_params_default.restype = None
    lib.vi_ctx_create.argtypes = [C.c_int, P(vp)]
    lib.vi_ctx_destroy.argtypes = [vp]
    lib.vi_ctx_destroy.restype = None
    lib.vi_set_grid.argtypes = [vp, vp, C.c_int]
    lib.vi_set_exclusions.argtypes = [vp, vp, C.c_int]
    lib.vi_set_ref_centroids.argtypes = [vp, vp, C.c_int, C.c_int]
    lib.vi_unit_pixels.argtypes = [vp]
    lib.vi_unit_pixels.restype = i64
    lib.vi_unit_offsets.argtypes = [vp, vp]
    lib.vi_host_upload_bytes.argtypes = [vp, C.c_int, i64]
    lib.vi_host_upload_bytes.restype = i64
    lib.vi_inspect_batch.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i64, i64, P(ViParams), vp, vp, vp, vp, vp]
    lib.vi_inspect_batch_host.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i64, i64, P(ViParams), vp, vp, vp]
    lib.vi_inspect_batch_host_fmt.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i64, i64, P(ViParams), C.c_int, vp, vp, vp]
    lib.vi_inspect_batch_host_blobs.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i64, i64, P(ViParams), C.c_int, vp, vp, vp,
                                                vp, C.c_int]
    lib.vi_segment_batch.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i64, i64, P(ViParams), vp, vp, vp]
    lib.vi_segment_batch_host.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i64, i64, P(ViParams), C.c_int, vp, vp]
    lib.vi_set_packed_mask_output.argtypes = [vp, vp, vp]
    lib.vi_set_defect_blob_output.argtypes = [vp, vp, C.c_int]
    lib.vi_packed_mask_bytes.argtypes = [vp]
    lib.vi_packed_mask_bytes.restype = i64
    lib.vi_packed_mask_offsets.argtypes = [vp, vp]
    lib.vi_peer_table_create.argtypes = [vp, i64, P(vp), vp]
    lib.vi_peer_table_open.argtypes = [vp, vp, P(vp)]
    lib.vi_peer_table_close.argtypes = [vp, vp]
    lib.vi_peer_table_destroy.argtypes = [vp, vp]
    lib.vi_peer_table_read.argtypes = [vp, vp, i64, vp]
    lib.vi_set_record_peers.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int]
    lib.vi_segment_cell.argtypes = [vp, vp, C.c_int, C.c_int, P(ViParams), vp, P(i32)]
    lib.vi_fill_internal_holes.argtypes = [vp, vp, C.c_int, C.c_int, vp]
    lib.vi_mask_stats.argtypes = [vp, vp, C.c_int, C.c_int, P(i64), P(i64), P(i64)]
    lib.vi_erode_square.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, vp]
    lib.vi_label_components.argtypes = [vp, vp, C.c_int, C.c_int, vp, P(i32), P(i32), P(i64), P(i64), P(i64)]
    lib.vi_debug_set_profile.argtypes = [vp, vp]
    lib.vi_debug_check_word.argtypes = [vp, P(C.c_uint32)]
    lib.vi_debug_fastdiv_check.argtypes = [vp, i64, C.c_uint64, P(i64)]
    lib.vi_debug_otsu.argtypes = [vp, vp, vp, C.c_int, vp]
    lib.vi_debug_rank_residual.argtypes = [vp, vp, vp, C.c_int, C.c_int, P(C.c_int), C.c_int, C.c_int, C.c_int, C.c_int, vp,
                                           P(C.c_int)]
    lib.vi_detect_defects.argtypes = [vp, vp, vp, C.c_int, C.c_int, P(ViParams), vp, P(i32), vp]
    lib.vi_debug_adaptive_taps.argtypes = [C.c_int, vp]
    lib.vi_set_seg_stats_output.argtypes = [vp, vp]
    lib.vi_ingest_argb32.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i64, i64, vp, i64, i64, vp]
    lib.vi_ingest_gray16.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, i64, i64, vp, i64, i64, vp]
    for n in EXPORTS:
        f = getattr(lib, n)
        if n not in ("vi_last_error", "vi_params_default", "vi_ctx_destroy", "vi_unit_pixels", "vi_version", "vi_host_upload_bytes",
                     "vi_packed_mask_bytes"):
            f.restype = C.c_int
    _lib = lib
    return lib


def check(rc):
    if rc != VI_OK:
        raise ViError(rc, load().vi_last_error().decode("utf-8", "replace"))


def default_params(**kw):
    p = ViParams()
    load().vi_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise TypeError(f"unknown parameter {k!r}")
        # the reference's combo-box strings (indexing_ui.py:800, :871); unknown strings take the default branch
        if k == "seg_method" and isinstance(v, str):
            v = 1 if v == "adaptive" else 0
        if k == "defect_method" and isinstance(v, str):
            v = 1 if v == "canny" else 0
        setattr(p, k, v)
    return p
