"""Host side of the B200 inspection path: a thin object over the C ABI.

`Inspector` owns one `vi_ctx` (one per process and device).  The batch call
takes device-resident frames (torch tensors -- PyTorch only supplies device
memory and streams); `inspect_batch_host` takes host arrays and pipelines
upload / compute / download inside the library."""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import BLOB_DTYPE, RECORD_DTYPE, ViExcl, check, default_params
from .grid import Grid, exclusions_to_table


def _u8c(a, name):
    a = np.ascontiguousarray(a)
    if a.dtype != np.uint8:
        raise TypeError(f"{name} must be uint8, got {a.dtype}")
    return a


class Inspector:
    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        check(self._lib.vi_ctx_create(int(device), C.byref(self._ctx)))
        self.device = int(device)
        self.n_units = 0
        self.unit_pixels = 0
        self.offsets = np.zeros(1, np.int64)
        self.shapes = []
        self.packed_bytes = 0
        self.packed_offsets = np.zeros(1, np.int64)

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.vi_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- configuration ---------------------------------------------------------
    def set_grid(self, rects: Sequence[Sequence[int]]):
        r = np.ascontiguousarray(np.asarray(rects, dtype=np.int32).reshape(-1, 4))
        check(self._lib.vi_set_grid(self._ctx, r.ctypes.data, int(r.shape[0])))
        self.n_units = int(r.shape[0])
        self.unit_pixels = int(self._lib.vi_unit_pixels(self._ctx))
        self.offsets = np.zeros(self.n_units + 1, np.int64)
        check(self._lib.vi_unit_offsets(self._ctx, self.offsets.ctypes.data))
        self.shapes = [(int(h), int(w)) for _, _, w, h in r]
        self.packed_bytes = int(self._lib.vi_packed_mask_bytes(self._ctx))
        self.packed_offsets = np.zeros(self.n_units + 1, np.int64)
        check(self._lib.vi_packed_mask_offsets(self._ctx, self.packed_offsets.ctypes.data))

    def set_exclusions(self, exclusions):
        rows = exclusions_to_table(exclusions or [])
        arr = (ViExcl * max(1, len(rows)))()
        for i, (s, a, b, c, d) in enumerate(rows):
            arr[i] = ViExcl(s, a, b, c, d)
        check(self._lib.vi_set_exclusions(self._ctx, C.cast(arr, C.c_void_p), len(rows)))

    def set_ref_centroids(self, ref_centroids: Optional[dict], is_reference: bool = False):
        """ref_centroids: {list position: (cx, cy)} (grid JSON v2) or None."""
        if not ref_centroids:
            check(self._lib.vi_set_ref_centroids(self._ctx, None, 0, int(bool(is_reference))))
            return
        tab = np.full((self.n_units, 2), np.nan, np.float64)
        for k, v in ref_centroids.items():
            if 0 <= int(k) < self.n_units:
                tab[int(k)] = (float(v[0]), float(v[1]))
        check(self._lib.vi_set_ref_centroids(self._ctx, tab.ctypes.data, self.n_units, int(bool(is_reference))))

    def configure(self, grid: Grid, is_reference: bool = False):
        self.set_grid(grid.rects)
        self.set_exclusions(grid.exclusions)
        self.set_ref_centroids(grid.ref_centroids, is_reference)

    # ---- batch calls -------------------------------------------------------------
    @staticmethod
    def _check_out(t, name, dev, dtype, numel):
        """A caller-supplied output tensor must be on the frames' device, contiguous, of the right type and size."""
        if t is None:
            return
        if not t.is_cuda or t.device != dev:
            raise ValueError(f"{name} must live on {dev}, got {t.device}")
        if t.dtype != dtype:
            raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
        if not t.is_contiguous():
            raise ValueError(f"{name} must be contiguous")
        if t.numel() < numel:
            raise ValueError(f"{name} holds {t.numel()} elements, the batch needs {numel}")

    def inspect_batch(self, frames, params=None, seg_masks=None, defect_masks=None, records=None, labels=None,
                      stream=None, seg_stats=None, seg_bits=None, defect_bits=None, defect_blobs=None):
        """frames: CUDA uint8 tensor [n, H, W] (row stride may exceed W).  Returns
        (records, seg_masks, defect_masks) as CUDA tensors (records: uint8 [n*units, 64]);
        asynchronous on `stream` (default: torch's current stream).
        defect_blobs: optional CUDA uint8 [n*units, K, 40] (1 <= K <= 1024): row uid gets the first min(n_kept, K) kept
        defect components of that unit (BLOB_DTYPE, raster order of their first pixel); later entries are not written."""
        import torch
        if not frames.is_cuda or frames.dtype != torch.uint8 or frames.dim() != 3:
            raise TypeError("frames must be a CUDA uint8 tensor [n, H, W]")
        if frames.stride(2) != 1:
            raise ValueError("frames must be contiguous along x")
        n, H, W = frames.shape
        dev = frames.device
        if dev.index != self.device:
            raise ValueError(f"frames are on {dev}, this Inspector drives cuda:{self.device}")
        total = n * self.unit_pixels
        self._check_out(seg_masks, "seg_masks", dev, torch.uint8, total)
        self._check_out(defect_masks, "defect_masks", dev, torch.uint8, total)
        self._check_out(records, "records", dev, torch.uint8, n * self.n_units * 64)
        self._check_out(labels, "labels", dev, torch.int32, total)
        self._check_out(seg_stats, "seg_stats", dev, torch.int64, n * self.n_units * 3)
        self._check_out(seg_bits, "seg_bits", dev, torch.uint8, n * self.packed_bytes)
        self._check_out(defect_bits, "defect_bits", dev, torch.uint8, n * self.packed_bytes)
        k_blobs = 0
        if defect_blobs is not None:
            if defect_blobs.dim() != 3 or defect_blobs.shape[2] != BLOB_DTYPE.itemsize:
                raise ValueError(f"defect_blobs must be [n*units, K, {BLOB_DTYPE.itemsize}]")
            k_blobs = int(defect_blobs.shape[1])
            self._check_out(defect_blobs, "defect_blobs", dev, torch.uint8, n * self.n_units * k_blobs * BLOB_DTYPE.itemsize)
        if seg_masks is None:
            seg_masks = torch.empty(total, dtype=torch.uint8, device=dev)
        if defect_masks is None:
            defect_masks = torch.empty(total, dtype=torch.uint8, device=dev)
        if records is None:
            records = torch.empty((n * self.n_units, 64), dtype=torch.uint8, device=dev)
        st = stream if stream is not None else torch.cuda.current_stream(dev)
        p = params if params is not None else default_params()
        # seg_stats: optional CUDA int64 [n*units, 3] (area, sum x, sum y of each final seg mask: the CSV export's numbers)
        check(self._lib.vi_set_seg_stats_output(self._ctx, seg_stats.data_ptr() if seg_stats is not None else None))
        # seg_bits / defect_bits: optional CUDA uint8 [n * packed_bytes]: the masks as 1 bit per pixel (PNG scanline order)
        check(self._lib.vi_set_packed_mask_output(self._ctx, seg_bits.data_ptr() if seg_bits is not None else None,
                                                  defect_bits.data_ptr() if defect_bits is not None else None))
        check(self._lib.vi_set_defect_blob_output(self._ctx, defect_blobs.data_ptr() if defect_blobs is not None else None,
                                                  k_blobs))
        check(self._lib.vi_inspect_batch(
            self._ctx, frames.data_ptr(), int(n), int(W), int(H), int(frames.stride(1)),
            int(frames.stride(0)) if n > 1 else int(frames.stride(1)) * int(H),
            C.byref(p), seg_masks.data_ptr(), defect_masks.data_ptr(),
            labels.data_ptr() if labels is not None else None, records.data_ptr(), C.c_void_p(st.cuda_stream)))
        return records, seg_masks, defect_masks

    def segment_batch(self, frames, params=None, seg_masks=None, records=None, stream=None, seg_stats=None, seg_bits=None):
        """run_segmentation_all for every unit of every frame, without the defect detector.  frames as for
        `inspect_batch`; returns (records, seg_masks) as CUDA tensors, asynchronous on `stream`.  Records carry otsu_t,
        seg_area, dx, dy, cx, cy (the pre-exclusion centroid: `grid.ref_centroids_from_records`) and status
        STATUS_SEGMENTED; the detector's fields are 0.  seg_stats / seg_bits: optional outputs as in `inspect_batch`."""
        import torch
        if not frames.is_cuda or frames.dtype != torch.uint8 or frames.dim() != 3:
            raise TypeError("frames must be a CUDA uint8 tensor [n, H, W]")
        if frames.stride(2) != 1:
            raise ValueError("frames must be contiguous along x")
        n, H, W = frames.shape
        dev = frames.device
        if dev.index != self.device:
            raise ValueError(f"frames are on {dev}, this Inspector drives cuda:{self.device}")
        total = n * self.unit_pixels
        self._check_out(seg_masks, "seg_masks", dev, torch.uint8, total)
        self._check_out(records, "records", dev, torch.uint8, n * self.n_units * 64)
        self._check_out(seg_stats, "seg_stats", dev, torch.int64, n * self.n_units * 3)
        self._check_out(seg_bits, "seg_bits", dev, torch.uint8, n * self.packed_bytes)
        if seg_masks is None:
            seg_masks = torch.empty(total, dtype=torch.uint8, device=dev)
        if records is None:
            records = torch.empty((n * self.n_units, 64), dtype=torch.uint8, device=dev)
        st = stream if stream is not None else torch.cuda.current_stream(dev)
        p = params if params is not None else default_params()
        check(self._lib.vi_set_seg_stats_output(self._ctx, seg_stats.data_ptr() if seg_stats is not None else None))
        check(self._lib.vi_set_packed_mask_output(self._ctx, seg_bits.data_ptr() if seg_bits is not None else None, None))
        check(self._lib.vi_segment_batch(
            self._ctx, frames.data_ptr(), int(n), int(W), int(H), int(frames.stride(1)),
            int(frames.stride(0)) if n > 1 else int(frames.stride(1)) * int(H),
            C.byref(p), seg_masks.data_ptr(), records.data_ptr(), C.c_void_p(st.cuda_stream)))
        return records, seg_masks

    # ---- frame ingest (device) -------------------------------------------------------
    def ingest_argb32(self, frames_bgra, out=None, stream=None):
        """QImage ARGB32 frames (CUDA uint8 [n, H, W, 4], bytes B,G,R,A) -> mono CUDA uint8 [n, H, W], the reference's
        `qimage_to_gray_array` (segmentation.py:15-23) for whole frames on the device."""
        import torch
        f = frames_bgra
        if not f.is_cuda or f.dtype != torch.uint8 or f.dim() != 4 or f.shape[3] != 4 or f.stride(3) != 1 or f.stride(2) != 4:
            raise TypeError("frames must be a CUDA uint8 tensor [n, H, W, 4] with packed pixels")
        n, H, W, _ = f.shape
        if out is None:
            out = torch.empty((n, H, W), dtype=torch.uint8, device=f.device)
        st = stream if stream is not None else torch.cuda.current_stream(f.device)
        check(self._lib.vi_ingest_argb32(self._ctx, f.data_ptr(), int(n), int(W), int(H), int(f.stride(1)),
                                         int(f.stride(0)) if n > 1 else int(f.stride(1)) * int(H), out.data_ptr(),
                                         int(out.stride(1)), int(out.stride(0)) if n > 1 else int(out.stride(1)) * int(H),
                                         C.c_void_p(st.cuda_stream)))
        return out

    def ingest_gray16(self, frames_u16, out=None, stream=None):
        """16-bit mono frames (CUDA int16/uint16 [n, H, W]) -> mono CUDA uint8 with the reference's loader rule
        `(arr / 256).astype(uint8)` (indexing_ui.py:153-155)."""
        import torch
        f = frames_u16
        if not f.is_cuda or f.element_size() != 2 or f.dim() != 3 or f.stride(2) != 1:
            raise TypeError("frames must be a CUDA 16-bit tensor [n, H, W]")
        n, H, W = f.shape
        if out is None:
            out = torch.empty((n, H, W), dtype=torch.uint8, device=f.device)
        st = stream if stream is not None else torch.cuda.current_stream(f.device)
        check(self._lib.vi_ingest_gray16(self._ctx, f.data_ptr(), int(n), int(W), int(H), int(f.stride(1)) * 2,
                                         (int(f.stride(0)) if n > 1 else int(f.stride(1)) * int(H)) * 2, out.data_ptr(),
                                         int(out.stride(1)), int(out.stride(0)) if n > 1 else int(out.stride(1)) * int(H),
                                         C.c_void_p(st.cuda_stream)))
        return out

    def inspect_batch_host(self, frames: np.ndarray, params=None, want_masks=True, out=None, mask_format="bytes",
                           max_blobs=0):
        """frames: host uint8 [n, H, W] (numpy, pageable or pinned -- e.g. a torch pin_memory tensor's .numpy(); either
        way the rows the grid covers are copied to the device).  mask_format: "bytes" (0/255, the reference's masks), "packed"
        (1 bit per pixel, see `unpack_masks`) or "none" (records only).
        Returns (records structured array, seg_masks u8 | None, defect_masks u8 | None).  With max_blobs = K > 0 a 4th
        element follows: the kept defect components, BLOB_DTYPE [n, units, K], of which the first min(n_kept, K) of each
        unit are valid (`kept_blobs`)."""
        frames = _u8c(frames, "frames")
        if frames.ndim != 3:
            raise ValueError("frames must be [n, H, W]")
        n, H, W = frames.shape
        fmt = {"bytes": _lib.MASKS_BYTES, "packed": _lib.MASKS_PACKED, "none": _lib.MASKS_NONE}[mask_format]
        if not want_masks:
            fmt = _lib.MASKS_NONE
        per_image = {_lib.MASKS_BYTES: self.unit_pixels, _lib.MASKS_PACKED: self.packed_bytes, _lib.MASKS_NONE: 0}[fmt]
        total = n * per_image
        if out is not None:
            rec, seg, dfm = out
            for nm, b in (("seg", seg), ("defect", dfm)):
                if b is not None and fmt != _lib.MASKS_NONE and (b.dtype != np.uint8 or not b.flags.c_contiguous or b.size < total):
                    raise ValueError(f"out {nm} buffer must be contiguous uint8 with at least {total} bytes")
            if rec.dtype != RECORD_DTYPE or not rec.flags.c_contiguous or rec.size < n * self.n_units:
                raise ValueError("out records buffer must be a contiguous RECORD_DTYPE array of n * units entries")
        else:
            rec = np.empty(n * self.n_units, RECORD_DTYPE)
            seg = np.empty(total, np.uint8) if fmt != _lib.MASKS_NONE else None
            dfm = np.empty(total, np.uint8) if fmt != _lib.MASKS_NONE else None
        if fmt == _lib.MASKS_NONE:
            seg = dfm = None
        p = params if params is not None else default_params()
        if max_blobs:
            if not 1 <= int(max_blobs) <= _lib.MAX_BLOBS_PER_UNIT:
                raise ValueError(f"max_blobs must be in 1..{_lib.MAX_BLOBS_PER_UNIT}, got {max_blobs}")
            blobs = np.empty((n, self.n_units, int(max_blobs)), BLOB_DTYPE)
            check(self._lib.vi_inspect_batch_host_blobs(
                self._ctx, frames.ctypes.data, int(n), int(W), int(H), int(W), int(H) * int(W), C.byref(p), fmt,
                seg.ctypes.data if seg is not None else None, dfm.ctypes.data if dfm is not None else None,
                rec.ctypes.data, blobs.ctypes.data, int(max_blobs)))
            return rec, seg, dfm, blobs
        check(self._lib.vi_inspect_batch_host_fmt(
            self._ctx, frames.ctypes.data, int(n), int(W), int(H), int(W), int(H) * int(W), C.byref(p), fmt,
            seg.ctypes.data if seg is not None else None, dfm.ctypes.data if dfm is not None else None,
            rec.ctypes.data))
        return rec, seg, dfm

    def segment_batch_host(self, frames: np.ndarray, params=None, mask_format="bytes"):
        """`segment_batch` from and to host arrays (frames uint8 [n, H, W]), pipelined as `inspect_batch_host` is.
        mask_format: "bytes", "packed" or "none".  Returns (records structured array, seg_masks u8 | None)."""
        frames = _u8c(frames, "frames")
        if frames.ndim != 3:
            raise ValueError("frames must be [n, H, W]")
        n, H, W = frames.shape
        fmt = {"bytes": _lib.MASKS_BYTES, "packed": _lib.MASKS_PACKED, "none": _lib.MASKS_NONE}[mask_format]
        per_image = {_lib.MASKS_BYTES: self.unit_pixels, _lib.MASKS_PACKED: self.packed_bytes, _lib.MASKS_NONE: 0}[fmt]
        rec = np.empty(n * self.n_units, RECORD_DTYPE)
        seg = np.empty(n * per_image, np.uint8) if fmt != _lib.MASKS_NONE else None
        p = params if params is not None else default_params()
        check(self._lib.vi_segment_batch_host(
            self._ctx, frames.ctypes.data, int(n), int(W), int(H), int(W), int(H) * int(W), C.byref(p), fmt,
            seg.ctypes.data if seg is not None else None, rec.ctypes.data))
        return rec, seg

    def kept_blobs(self, records, blobs, image, unit):
        """The valid kept-component entries of one (image, unit): records (RECORD_DTYPE, [n*units] or [n, units]) and a
        blob table from either batch call (BLOB_DTYPE [n, units, K], or the device table's uint8 [n*units, K, 40] copied
        to the host).  Returns a BLOB_DTYPE array of min(n_kept, K) entries, unit-local coordinates."""
        b = np.asarray(blobs)
        if b.dtype != BLOB_DTYPE:
            b = np.ascontiguousarray(b).view(BLOB_DTYPE)[..., 0]
        uid = int(image) * self.n_units + int(unit)
        b = b.reshape(-1, b.shape[-1])
        n_kept = int(np.asarray(records).reshape(-1)[uid]['n_kept'])
        return b[uid, :min(n_kept, b.shape[1])]

    def unpack_masks(self, packed, image=0):
        """One image's packed-bit mask block (mask_format="packed") as a list of (h, w) uint8 0/255 arrays."""
        base = image * self.packed_bytes
        out = []
        for u, (h, w) in enumerate(self.shapes):
            blk = np.asarray(packed[base + self.packed_offsets[u]: base + self.packed_offsets[u + 1]]).reshape(h, -1)
            out.append(np.unpackbits(blk, axis=1)[:, :w] * np.uint8(255))
        return out

    def split_masks(self, flat, image=0):
        """View one image's packed mask block as a list of (h, w) arrays."""
        base = image * self.unit_pixels
        return [flat[base + self.offsets[u]: base + self.offsets[u + 1]].reshape(self.shapes[u])
                for u in range(self.n_units)]

    # ---- per-unit compat calls (host arrays) ----------------------------------------
    def segment_cell(self, gray, params=None, return_threshold=False):
        gray = _u8c(gray, "gray")
        h, w = gray.shape
        out = np.empty((h, w), np.uint8)
        t = C.c_int32(0)
        p = params if params is not None else default_params()
        check(self._lib.vi_segment_cell(self._ctx, gray.ctypes.data, h, w, C.byref(p), out.ctypes.data, C.byref(t)))
        return (out, int(t.value)) if return_threshold else out

    def fill_internal_holes(self, mask):
        mask = _u8c(mask, "mask")
        h, w = mask.shape
        out = np.empty((h, w), np.uint8)
        check(self._lib.vi_fill_internal_holes(self._ctx, mask.ctypes.data, h, w, out.ctypes.data))
        return out

    def mask_sums(self, mask):
        mask = _u8c(mask, "mask")
        h, w = mask.shape
        a, sx, sy = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        check(self._lib.vi_mask_stats(self._ctx, mask.ctypes.data, h, w, C.byref(a), C.byref(sx), C.byref(sy)))
        return int(a.value), int(sx.value), int(sy.value)

    def erode_square(self, mask, r):
        mask = _u8c(mask, "mask")
        h, w = mask.shape
        out = np.empty((h, w), np.uint8)
        check(self._lib.vi_erode_square(self._ctx, mask.ctypes.data, h, w, int(r), out.ctypes.data))
        return out

    def label_components(self, mask, want_labels=True):
        """-> dict(labels int32[h,w] raster-canonical | None, n, best_label, best_area, centroid | None)"""
        mask = _u8c(mask, "mask")
        h, w = mask.shape
        lab = np.empty((h, w), np.int32) if want_labels else None
        n, best = C.c_int32(0), C.c_int32(0)
        a, sx, sy = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        check(self._lib.vi_label_components(self._ctx, mask.ctypes.data, h, w,
                                            lab.ctypes.data if lab is not None else None, C.byref(n), C.byref(best),
                                            C.byref(a), C.byref(sx), C.byref(sy)))
        cen = (sx.value / a.value, sy.value / a.value) if a.value > 0 else None
        return dict(labels=lab, n=int(n.value), best_label=int(best.value), best_area=int(a.value), centroid=cen)

    def detect_defects(self, gray, seg_mask, params=None, return_record=False):
        gray = _u8c(gray, "gray")
        seg_mask = _u8c(seg_mask, "seg_mask")
        if gray.shape != seg_mask.shape:
            raise ValueError("gray and seg_mask must have the same shape")   # the reference rescales; this app never needs to
        h, w = gray.shape
        out = np.empty((h, w), np.uint8)
        found = C.c_int32(0)
        rec = np.zeros(1, RECORD_DTYPE)
        p = params if params is not None else default_params()
        check(self._lib.vi_detect_defects(self._ctx, gray.ctypes.data, seg_mask.ctypes.data, h, w, C.byref(p),
                                          out.ctypes.data, C.byref(found), rec.ctypes.data))
        res = out if found.value else None
        return (res, rec[0]) if return_record else res


_default = {}


def default_inspector(device: Optional[int] = None) -> Inspector:
    """Lazily created per-process context (the UI calls from one thread only)."""
    import os
    if device is None:
        device = int(os.environ.get("VI_B200_DEVICE", "0"))
    if device not in _default:
        _default[device] = Inspector(device)
    return _default[device]
