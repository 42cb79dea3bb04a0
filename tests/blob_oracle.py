"""cv2 oracle of the kept-defect-component table (vi_set_defect_blob_output).

`kept_defect_blobs` runs the detector of oracle/ref_cv2.detect_defects (indexing_ui.py:1471-1560) up to its contour
loop and describes every contour that passes the area filter (:1551-1558) instead of only drawing it: its bounding box,
2 * contourArea, and the count and mean x / y of the pixels that drawContours(FILLED) paints for it.  The list is in
raster order of the first painted pixel, the order of the library's table."""
import cv2
import numpy as np

from oracle import ref_cv2 as R

BLOB_FIELDS = ("x", "y", "w", "h", "area", "area2", "cx", "cy")


def kept_contours(gray, seg_mask, method='threshold', threshold=24, min_area=20, erode_px=6):
    """The kept contours of detect_defects, in findContours order ([] where the detector returns early)."""
    info = {}
    if R.detect_defects(gray, seg_mask, method, threshold, min_area, erode_px, info) is None:
        return []
    seg_bin = info.get('roi')
    thr = int(threshold)
    if method == 'threshold':                                     # the same steps as R.detect_defects
        bg = cv2.medianBlur(gray, 21)
        _, mask = cv2.threshold(cv2.absdiff(gray, bg), thr, 255, cv2.THRESH_BINARY)
        if seg_bin is not None:
            mask = cv2.bitwise_and(mask, seg_bin)
        mask = cv2.morphologyEx(mask, cv2.MORPH_OPEN, cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (3, 3)), iterations=1)
    else:
        mask = cv2.Canny(gray, max(1, thr // 2), max(2, thr))
        if seg_bin is not None:
            mask = cv2.bitwise_and(mask, seg_bin)
    cnts, _ = cv2.findContours(mask.copy(), cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    seg_area = int((seg_bin > 0).sum()) if seg_bin is not None else int(gray.shape[0] * gray.shape[1])
    max_area = max(int(min_area), int(seg_area * 0.98))
    kept = [c for c in cnts if int(min_area) <= cv2.contourArea(c) <= max_area]
    assert len(kept) == info['n_kept']
    return kept


def describe(contours, shape):
    """One dict per contour (BLOB_FIELDS plus the painted pixel set as flat indices), sorted by first painted pixel."""
    out = []
    for c in contours:
        # painted on the contour's bounding rectangle (drawContours never paints outside it; test_blob_oracle checks
        # the box against the whole-unit drawing)
        bx, by, bw, bh = cv2.boundingRect(c)
        d = np.zeros((bh, bw), np.uint8)
        cv2.drawContours(d, [c], -1, 255, -1, offset=(-bx, -by))
        ys, xs = np.nonzero(d)
        ys, xs = ys + by, xs + bx
        out.append(dict(x=int(xs.min()), y=int(ys.min()), w=int(xs.max() - xs.min() + 1), h=int(ys.max() - ys.min() + 1),
                        area=int(xs.size), area2=int(2 * cv2.contourArea(c)), cx=float(xs.mean()), cy=float(ys.mean()),
                        pixels=ys.astype(np.int64) * shape[1] + xs, contour=c))
    out.sort(key=lambda b: int(b['pixels'][0]))
    return out


def kept_defect_blobs(gray, seg_mask, method='threshold', threshold=24, min_area=20, erode_px=6):
    return describe(kept_contours(gray, seg_mask, method, threshold, min_area, erode_px), gray.shape)


def params_kw(rp):
    """kept_defect_blobs' keyword arguments from an R.Params."""
    return dict(method=rp.defect_method, threshold=rp.threshold, min_area=rp.min_area, erode_px=rp.erode_px)


def assert_blobs_equal(got, want, ctx):
    """The library's entries (BLOB_DTYPE) against the oracle's, field for field; cx / cy bit for bit."""
    assert len(got) == len(want), (ctx, len(got), len(want))
    for j, (g, o) in enumerate(zip(got, want)):
        for f in ("x", "y", "w", "h", "area", "area2"):
            assert int(g[f]) == o[f], (ctx, j, f, int(g[f]), o[f])
        for f in ("cx", "cy"):
            assert np.float64(g[f]).view(np.int64) == np.float64(o[f]).view(np.int64), (ctx, j, f, float(g[f]), o[f])
