"""Drop-in for the reference's ``segmentation.py`` (same names, same signatures,
same error behaviour) running on the B200 through the C ABI.

``import segmentation`` in the reference UI keeps working when this module is put
in its place (INTEGRATION.md).  New in the same style: ``detect_defects`` (the
compute body of ``MainWindow._detect_defects_on_pix``, indexing_ui.py:1471-1572,
minus Qt), ``inspect_batch`` and ``segment_batch``.  No CPU fallback: without a CUDA device or the
built extension every compute call raises."""
from __future__ import annotations

import numpy as np

from ._lib import default_params
from .api import default_inspector

try:  # same guarded import as the reference (segmentation.py:4-7)
    from PyQt6.QtGui import QImage
except Exception:  # pragma: no cover - PyQt6 is absent on the build and GPU boxes
    QImage = None


def qimage_to_gray_array(qimg):
    """segmentation.py:10-24 -- host-side Qt plumbing, kept as is.  The gray value is
    (R*3735 + G*19235 + B*9798 + 16384) >> 15 on the byte order the reference
    feeds to cv2 (R/B swapped, SURVEY A.1); identity for mono images."""
    if QImage is None:
        raise RuntimeError("PyQt6 is required for qimage_to_gray_array() in improved_UI")
    qimg = qimg.convertToFormat(QImage.Format.Format_ARGB32)
    ptr = qimg.bits()
    byte_count = getattr(qimg, "sizeInBytes", None)
    byte_count = byte_count() if callable(byte_count) else qimg.byteCount()
    ptr.setsize(int(byte_count))
    arr = np.frombuffer(ptr, np.uint8).reshape((qimg.height(), qimg.width(), 4)).astype(np.uint32)
    b, g, r = arr[:, :, 0], arr[:, :, 1], arr[:, :, 2]
    return ((r * 3735 + g * 19235 + b * 9798 + 16384) >> 15).astype(np.uint8)


def fill_internal_holes(mask):
    """segmentation.py:27-72."""
    if mask is None:
        return mask
    if mask.ndim != 2:
        raise ValueError('fill_internal_holes expects a 2D mask')
    if mask.shape[0] == 0 or mask.shape[1] == 0:
        return (mask > 0).astype(np.uint8) * 255
    m = mask if mask.dtype == np.uint8 else (mask > 0).astype(np.uint8)
    return default_inspector().fill_internal_holes(m)


def segment_cell(gray, method='otsu', adapt_block=51, adapt_C=10, gaussian_blur=3, morph_kernel=3):
    """segmentation.py:75-100.  Returns a fresh, writable uint8 0/255 array; `gray`
    is not modified.  Unknown `method` strings fall back to Otsu (:87-89)."""
    p = default_params(
        seg_method=1 if method == 'adaptive' else 0,
        adapt_block=int(adapt_block), adapt_C=int(adapt_C),
        gaussian_blur=int(gaussian_blur) if gaussian_blur else 0,
        morph_kernel=int(morph_kernel) if morph_kernel else 0)
    return default_inspector().segment_cell(np.asarray(gray), p)


def mask_stats(mask):
    """segmentation.py:103-111."""
    m = np.asarray(mask)
    if m.dtype != np.uint8:
        m = (m > 0).astype(np.uint8)
    if m.size == 0:
        return {'area': 0, 'centroid': (0, 0)}
    area, sx, sy = default_inspector().mask_sums(m)
    if area == 0:
        return {'area': 0, 'centroid': (0, 0)}
    return {'area': int(area), 'centroid': (float(sx / area), float(sy / area))}


def detect_defects(gray, seg_mask, *, method='threshold', threshold=24, min_area=20, erode_px=6):
    """MainWindow._detect_defects_on_pix (indexing_ui.py:1471-1572) minus Qt:
    the defect mask (uint8 0/255) or None."""
    p = default_params(defect_method=1 if method == 'canny' else 0, threshold=int(threshold),
                       min_area=int(min_area), erode_px=int(erode_px))
    return default_inspector().detect_defects(np.asarray(gray), np.asarray(seg_mask), p)


def inspect_batch(frames, grid, params=None, is_reference=False):
    """run_segmentation_all + run_inspection (indexing_ui.py:2268-2338, :1669-1702)
    for every unit of every frame.  frames: uint8 [n, H, W] host array; grid: a
    vi_b200.grid.Grid.  Returns (records, seg_masks, defect_masks) with masks as
    per-image lists of (h, w) arrays."""
    insp = default_inspector()
    insp.configure(grid, is_reference=is_reference)
    rec, seg, dfm = insp.inspect_batch_host(np.asarray(frames), params)
    n = len(frames)
    return (rec.reshape(n, insp.n_units),
            [insp.split_masks(seg, i) for i in range(n)],
            [insp.split_masks(dfm, i) for i in range(n)])


def segment_batch(frames, grid, params=None, is_reference=False):
    """run_segmentation_all (indexing_ui.py:2203-2368) for every unit of every frame, without the defect detector.
    frames: uint8 [n, H, W] host array; grid: a vi_b200.grid.Grid.  Returns (records, seg_masks): records [n, units]
    (status STATUS_SEGMENTED; cx / cy feed `grid.ref_centroids_from_records`), masks as per-image lists of (h, w)
    arrays."""
    insp = default_inspector()
    insp.configure(grid, is_reference=is_reference)
    rec, seg = insp.segment_batch_host(np.asarray(frames), params)
    n = len(frames)
    return rec.reshape(n, insp.n_units), [insp.split_masks(seg, i) for i in range(n)]
