"""CPU ORACLE (test infrastructure, NOT product code) -- integer restatement.

cv2-free restatement (numpy + scipy.ndimage only) of every stage of the hot
path, in the contour-free form the CUDA kernels implement one-to-one
(SURVEY.md Appendix A).  ``tests/test_restate_vs_cv2.py`` proves each function
here equal to the cv2 arm (``oracle/ref_cv2.py``), which in turn is pinned to
the reference's own outputs (``tests/golden``).  The CUDA parity tests may then
use either arm.

Each function cites the reference call site it restates (file:line under
/root/reference) and the SURVEY appendix that states the equivalence.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import numpy as np
from scipy import ndimage as ndi

FLT_EPSILON = 1.1920928955078125e-07


# --------------------------------------------------------------------------- K2
_SMALL_GAUSS = {
    1: [1.0],
    3: [0.25, 0.5, 0.25],
    5: [0.0625, 0.25, 0.375, 0.25, 0.0625],
    7: [0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125],
}


def gaussian_kernel_q8(k: int):
    """8.8 fixed-point taps OpenCV uses for uint8 GaussianBlur(k, sigma=0)
    (segmentation.py:80; SURVEY A.2): double kernel (hard-coded for k<=7,
    else exp(-x^2/2s^2) normalised, s = 0.3*((k-1)*0.5-1)+0.8), quantised
    outside-in with error diffusion, centre tap = 256 - rest."""
    if k in _SMALL_GAUSS:
        kern = list(_SMALL_GAUSS[k])
    else:
        sigma = ((k - 1) * 0.5 - 1) * 0.3 + 0.8
        s2 = -0.5 / (sigma * sigma)
        kern = [math.exp(s2 * (i - (k - 1) * 0.5) ** 2) for i in range(k)]
        tot = sum(kern)
        kern = [v * (1.0 / tot) for v in kern]
    q = [0] * k
    err = 0.0
    acc = 0
    for i in range(k // 2):
        adj = kern[i] * 256.0 + err
        v = int(round(adj))              # Python round == cvRound (half to even)
        err = adj - v
        q[i] = q[k - 1 - i] = v
        acc += v
    q[k // 2] = 256 - 2 * acc
    return q


def _reflect101(idx, n):
    if n == 1:
        return np.zeros_like(idx)
    p = 2 * (n - 1)
    idx = np.mod(idx, p)
    return np.where(idx >= n, p - idx, idx)


def gaussian_blur_u8(img, ksize: int):
    """cv2.GaussianBlur(img,(k,k),0) for uint8, BORDER_REFLECT_101, bit-exact
    (segmentation.py:78-80).  ksize as the reference passes it: 0 -> skip,
    even -> +1."""
    if not ksize or ksize <= 0:
        return img.copy()
    k = int(ksize) if ksize % 2 == 1 else int(ksize) + 1
    q = gaussian_kernel_q8(k)
    h, w = img.shape
    r = k // 2
    src = img.astype(np.int64)
    xs = _reflect101(np.arange(-r, w + r), w)
    hp = np.zeros((h, w), np.int64)
    for i in range(k):
        hp += q[i] * src[:, xs[i:i + w]]
    ys = _reflect101(np.arange(-r, h + r), h)
    vp = np.zeros((h, w), np.int64)
    for i in range(k):
        vp += q[i] * hp[ys[i:i + h], :]
    return ((vp + 32768) >> 16).astype(np.uint8)


# --------------------------------------------------------------------------- K3
def otsu_from_hist(hist) -> int:
    """The Otsu scan of cv2.threshold(...OTSU) in IEEE doubles, in OpenCV's
    operation order (segmentation.py:82; SURVEY A.3)."""
    hist = [int(v) for v in hist]
    n = sum(hist)
    scale = 1.0 / n
    mu = 0.0
    for i in range(256):
        mu += i * float(hist[i])
    mu *= scale
    mu1 = 0.0
    q1 = 0.0
    max_sigma = 0.0
    max_val = 0
    for i in range(256):
        p_i = hist[i] * scale
        mu1 *= q1
        q1 += p_i
        q2 = 1.0 - q1
        if min(q1, q2) < FLT_EPSILON or max(q1, q2) > 1.0 - FLT_EPSILON:
            continue
        mu1 = (mu1 + i * p_i) / q1
        mu2 = (mu - q1 * mu1) / q2
        sigma = q1 * q2 * (mu1 - mu2) * (mu1 - mu2)
        if sigma > max_sigma:
            max_sigma = sigma
            max_val = i
    return max_val


def _otsu_scan_rows(H, last=None):
    """otsu_from_hist on every row of H, scoring only bins <= last (per row) when given."""
    H = np.asarray(H, dtype=np.int64)
    Hf = np.ascontiguousarray(H.T).astype(np.float64)          # [256, n]: exact (counts < 2^53)
    n = H.shape[0]
    scale = 1.0 / Hf.sum(0)
    mu = np.zeros(n)
    for i in range(256):
        mu += i * Hf[i]
    mu *= scale
    mu1 = np.zeros(n)
    q1 = np.zeros(n)
    max_sigma = np.zeros(n)
    max_val = np.zeros(n, np.int64)
    with np.errstate(divide='ignore', invalid='ignore'):
        for i in range(256):
            p_i = Hf[i] * scale
            mu1 *= q1
            q1 = q1 + p_i
            q2 = 1.0 - q1
            ok = ~((np.minimum(q1, q2) < FLT_EPSILON) | (np.maximum(q1, q2) > 1.0 - FLT_EPSILON))
            if last is not None:
                ok &= i <= last
            m1 = (mu1 + i * p_i) / q1
            mu2 = (mu - q1 * m1) / q2
            sigma = q1 * q2 * (m1 - mu2) * (m1 - mu2)
            mu1 = np.where(ok, m1, mu1)
            better = ok & (sigma > max_sigma)
            max_sigma = np.where(better, sigma, max_sigma)
            max_val = np.where(better, i, max_val)
    return max_val


def otsu_from_hists(H) -> np.ndarray:
    """otsu_from_hist over the rows of H ([n, 256] counts, each row's sum >= 1), vectorised: the same float64
    operations in the same order on every row, so the same thresholds bit for bit."""
    return _otsu_scan_rows(H)


def otsu_kernel_model(H, slack: float = 0.0):
    """The two steps of the device Otsu (vi_pipeline.cuh) on the rows of H ([n, 256] counts, sums 1..2^24):
    otsu_approx_warp's float32 between-class variances from exact integer moments (IEEE division where the kernel
    uses __fdividef) give `last`, the last bin within 2e-5 of their maximum; otsu_scan is the reference scan scoring
    bins <= last only.  Bins whose lower class is below FLT_EPSILON of the pixels (n1 * 2^23 < N), which the
    reference skips, score 0, as do bins with an empty upper class.  Once the reference skips a lone darkest pixel
    at x0, its mu1 lacks that pixel's x0 / N for good, so every later variance is the one of lower-class moment
    m1 - x0.  slack > 0 lowers every variance by that fraction and raises the maximum by as much, so `last` is what a
    division off by that much could give at worst.
    Returns (t, last), int64 arrays."""
    H = np.asarray(H, dtype=np.int64)
    N = H.sum(1)[:, None]
    n1 = np.cumsum(H, 1)
    m1 = np.cumsum(H * np.arange(256), 1)
    n2 = N - n1
    # above 2^23 pixels a lone darkest pixel's split is skipped, and with it the step that adds its value to mu1
    x0 = np.argmax(H > 0, 1)[:, None]
    drop = np.where((np.take_along_axis(H, x0, 1) == 1) & (N > (1 << 23)), x0, 0)
    dd = m1[:, -1:] * n1 - N * (m1 - drop)                      # exact: |dd| < 2^56
    f = dd.astype(np.float32)
    den = n1.astype(np.float32) * n2.astype(np.float32)
    scored = ((n1 << 23) >= N) & (n2 > 0)
    with np.errstate(divide='ignore', invalid='ignore'):
        v = np.where(scored, (f * f) / den, np.float32(0))
    mx = v.max(1, keepdims=True)
    keep = np.float32(1) - np.float32(2e-5)
    if slack:
        ge = v.astype(np.float64) * (1.0 - slack) >= mx.astype(np.float64) * (1.0 + slack) * np.float64(keep)
    else:
        ge = v >= mx * keep
    lc = 255 - np.argmax(ge[:, ::-1], 1)
    last = np.where(mx[:, 0] > 0, lc, 255)
    return _otsu_scan_rows(H, last), last


def otsu_inv_mask(img) -> Tuple[int, np.ndarray]:
    t = otsu_from_hist(np.bincount(img.ravel(), minlength=256))
    return t, np.where(img > t, 0, 255).astype(np.uint8)


# --------------------------------------------------------------------------- K5/K9/K13
def ellipse_se(k: int):
    """cv2.getStructuringElement(MORPH_ELLIPSE,(k,k)) (segmentation.py:93,
    indexing_ui.py:1532; SURVEY A.5): row i spans [c-dx, c+dx] with
    dx = round_half_even(c*sqrt((r^2-dy^2)/r^2)), r=c=k//2, dy=i-r."""
    r = k // 2
    c = k // 2
    inv_r2 = 1.0 / (r * r) if r else 0.0
    se = np.zeros((k, k), np.uint8)
    for i in range(k):
        dy = i - r
        if abs(dy) <= r:
            dx = int(round(c * math.sqrt((r * r - dy * dy) * inv_r2)))
            j1 = max(c - dx, 0)
            j2 = min(c + dx + 1, k)
            se[i, j1:j2] = 1
    return se


def _morph(mask, se, op):
    """erode: min over SE offsets, out-of-crop = 255; dilate: max over the same
    (un-reflected) offsets, out-of-crop = 0.  Anchor (k//2, k//2)."""
    kh, kw = se.shape
    ay, ax = kh // 2, kw // 2
    h, w = mask.shape
    pad = 255 if op == 'erode' else 0
    p = np.full((h + kh, w + kw), pad, np.uint8)
    p[ay:ay + h, ax:ax + w] = mask
    out = np.full((h, w), pad, np.uint8)
    for j in range(kh):
        for i in range(kw):
            if se[j, i]:
                v = p[j:j + h, i:i + w]
                out = np.minimum(out, v) if op == 'erode' else np.maximum(out, v)
    return out


def morph_close_open(mask, k: int):
    """segmentation.py:91-95."""
    if not k or k <= 0:
        return mask
    se = ellipse_se(max(1, int(k)))
    m = _morph(_morph(mask, se, 'dilate'), se, 'erode')      # CLOSE
    return _morph(_morph(m, se, 'erode'), se, 'dilate')      # OPEN


def open_cross3(mask):
    """indexing_ui.py:1532."""
    se = ellipse_se(3)
    return _morph(_morph(mask, se, 'erode'), se, 'dilate')


def erode_square(mask, r: int):
    """cv2.erode(mask, None, iterations=r) == one (2r+1)^2 square erosion with
    out-of-crop = 255 (indexing_ui.py:1497; SURVEY A.5)."""
    if r <= 0:
        return mask.copy()
    return ndi.minimum_filter(mask, size=2 * r + 1, mode='constant', cval=255)


# --------------------------------------------------------------------------- K6
_CROSS = np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]], np.uint8)
_FULL = np.ones((3, 3), np.uint8)


def fill_holes_4bg(mask):
    """segmentation.py:27-72 == fill every background region that is not
    4-connected to a background pixel on the crop border (SURVEY A.6)."""
    m = mask > 0
    h, w = m.shape
    if h == 0 or w == 0:
        return (m * 255).astype(np.uint8)
    lab, n = ndi.label(~m, structure=_CROSS)
    border = np.zeros(n + 1, bool)
    for edge in (lab[0, :], lab[-1, :], lab[:, 0], lab[:, -1]):
        border[edge] = True
    border[0] = True
    holes = ~border[lab]
    return ((m | holes) * 255).astype(np.uint8)


# --------------------------------------------------------------------------- K7/K10
def label8(mask):
    """8-connected labels in raster order of first pixel (canonical form used
    for parity dumps, SURVEY A.7)."""
    lab, n = ndi.label(mask > 0, structure=_FULL)
    return lab.astype(np.int32), n


def largest_component(mask):
    """(best_label_mask, area, sum_x, sum_y) of the component cv2 would pick at
    indexing_ui.py:1505-1510 / :2240-2248: max area, ties -> smallest cv2 label
    == smallest 2x2-block key min((y//2)*ceil(w/2) + x//2) (SURVEY A.7)."""
    lab, n = label8(mask)
    if n == 0:
        return None
    h, w = lab.shape
    ys, xs = np.nonzero(lab)
    ls = lab[ys, xs]
    area = np.bincount(ls, minlength=n + 1)
    key = (ys // 2) * ((w + 1) // 2) + (xs // 2)
    minkey = np.full(n + 1, np.iinfo(np.int64).max, np.int64)
    np.minimum.at(minkey, ls, key)
    order = sorted(range(1, n + 1), key=lambda l: (-int(area[l]), int(minkey[l])))
    best = order[0]
    sel = ls == best
    return lab == best, int(area[best]), int(xs[sel].sum()), int(ys[sel].sum())


def largest_component_centroid(mask):
    r = largest_component(mask)
    if r is None:
        return None
    _, a, sx, sy = r
    return (sx / a, sy / a)


# --------------------------------------------------------------------------- K8
def apply_exclusions(mask, exclusions, dx, dy):
    """indexing_ui.py:2316-2338 with the circle as per-row integer half-widths."""
    h, w = mask.shape
    for e in exclusions:
        if e.get('shape') == 'rect':
            ex, ey = int(e.get('x', 0)) + dx, int(e.get('y', 0)) + dy
            x0, y0 = max(0, ex), max(0, ey)
            x1, y1 = min(w, ex + int(e.get('w', 0))), min(h, ey + int(e.get('h', 0)))
            if x1 > x0 and y1 > y0:
                mask[y0:y1, x0:x1] = 0
        else:
            cx, cy, r = int(e.get('cx', 0)) + dx, int(e.get('cy', 0)) + dy, int(e.get('r', 0))
            if r > 0:
                for y in range(max(0, cy - r), min(h, cy + r + 1)):
                    hw = math.isqrt(r * r - (y - cy) ** 2)
                    x0, x1 = max(0, cx - hw), min(w, cx + hw + 1)
                    if x1 > x0:
                        mask[y, x0:x1] = 0
    return mask


# --------------------------------------------------------------------------- K11/K12
def median21(gray, k: int = 21):
    """cv2.medianBlur(gray, 21): true median, BORDER_REPLICATE
    (indexing_ui.py:1522-1525; SURVEY A.9)."""
    r = k // 2
    p = np.pad(gray, r, mode='edge')
    win = np.lib.stride_tricks.sliding_window_view(p, (k, k)).reshape(gray.shape[0], gray.shape[1], k * k)
    rank = (k * k) // 2
    return np.partition(win, rank, axis=2)[:, :, rank].copy()


def residual_mask_direct(gray, thr: int):
    bg = median21(gray).astype(np.int32)
    return (np.abs(gray.astype(np.int32) - bg) > thr)


def box_count_le(gray, level: int, k: int = 21):
    """#(window <= level) for every pixel, replicate border."""
    r = k // 2
    ind = (np.pad(gray, r, mode='edge') <= level).astype(np.int32)
    s = np.cumsum(np.cumsum(ind, axis=0), axis=1)
    s = np.pad(s, ((1, 0), (1, 0)))
    h, w = gray.shape
    return s[k:k + h, k:k + w] - s[0:h, k:k + w] - s[k:k + h, 0:w] + s[0:h, 0:w]


def residual_mask_rank(gray, thr: int, levels, stats: Optional[dict] = None):
    """The kernels' formulation of `|gray - median21(gray)| > thr`
    (indexing_ui.py:1522-1527) without ever forming the median:

        med >  g+thr   <=>  #(window <= g+thr)   <= 220
        med <= g-thr-1 <=>  #(window <= g-thr-1) >= 221

    Counts C_k at a few fixed `levels` v_0<..<v_{K-1} bracket the median,
    v_{km-1} < med <= v_{km}; a pixel whose pivots are separated from the
    bracket is decided from the bracket alone, the rest ('ambiguous') get an
    exact rank count at their own pivot.  Exact for ANY level set."""
    levels = sorted(set(int(v) for v in levels))
    K = len(levels)
    g = gray.astype(np.int32)
    half = 221
    km = np.zeros(gray.shape, np.int32)
    for v in levels:
        km += (box_count_le(gray, v) < half)
    lo = np.array([-1] + levels, np.int32)[km]           # med > lo
    hi = np.array(levels + [255], np.int32)[km]          # med <= hi
    a = g + thr
    b = g - thr - 1
    d1_true = lo >= a
    d1_false = hi <= a
    d2_true = hi <= b
    d2_false = lo >= b
    sure = d1_true | d2_true
    amb1 = ~(d1_true | d1_false)
    amb2 = ~(d2_true | d2_false)
    amb = ~sure & (amb1 | amb2)
    out = sure.copy()
    if stats is not None:
        stats['ambiguous'] = int(amb.sum())
    if amb.any():
        pad = np.pad(gray, 10, mode='edge')
        for y, x in zip(*np.nonzero(amb)):
            win = pad[y:y + 21, x:x + 21]
            r = False
            if amb1[y, x]:
                r = r or int((win <= a[y, x]).sum()) <= 220
            if amb2[y, x]:
                r = r or int((win <= b[y, x]).sum()) >= 221
            out[y, x] = r
    return out


def _lattice_brackets(gray, thr: int, levels):
    """C_k at the cell centres ([K][ny][nx]) and each cell's bracket LO < med <= HI ([ny][nx])."""
    K = len(levels)
    h, w = gray.shape
    ny, nx = (h + 2) // 3, (w + 2) // 3
    # exact counts at virtual centres (3j+1, 3i+1): replicate padding also beyond the crop
    pad = np.pad(gray, ((10, 10 + 3), (10, 10 + 3)), mode='edge')
    cy = 3 * np.arange(ny) + 1
    cx = 3 * np.arange(nx) + 1
    centre = []
    for v in levels:
        ind = (pad <= v).astype(np.int32)
        s = np.pad(np.cumsum(np.cumsum(ind, axis=0), axis=1), ((1, 0), (1, 0)))
        centre.append(s[cy[:, None] + 21, cx[None, :] + 21] - s[cy[:, None], cx[None, :] + 21]
                      - s[cy[:, None] + 21, cx[None, :]] + s[cy[:, None], cx[None, :]])
    C = np.stack(centre)
    lo_idx = (C <= 178).sum(0)
    hi_idx = K - (C >= 263).sum(0)
    LO = np.array([-1] + levels, np.int32)[lo_idx]
    HI = np.array(levels + [255], np.int32)[hi_idx]
    return C, LO, HI


def lattice_stats(gray, thr: int, levels, roi=None, cell_gray=None) -> dict:
    """What the kernel's stage counts (vi_rank.cuh: rank_dirty_cell, rank_finish), from the twin's brackets:
      ambiguous        ambiguous pixels (of the ROI when one is given): neither defect nor clean for sure
      entries          list entries, one per open test of an ambiguous pixel:
                       [g < HI - thr] + [g > LO + thr + 1]
      centre_counts    [K][ny][nx] C_k at the cell centres
      dirty_roi_cells  cells whose gray min or max leaves the clean range [HI - thr, LO + thr + 1]
                       and that hold a ROI pixel (every such cell without a ROI)
      codes            [16] bracket codes n179 * 4 + n263 of those cells (n263 <= n179: ten occur)
    The cell min / max are taken over `cell_gray` ([3 ny][3 nx], the bytes the kernel's min / max pass reads)
    when given, else over the crop with replicated rows and columns."""
    levels = sorted(int(v) for v in levels)
    h, w = gray.shape
    ny, nx = (h + 2) // 3, (w + 2) // 3
    C, LO, HI = _lattice_brackets(gray, thr, levels)
    g = gray.astype(np.int32)
    LOp = np.repeat(np.repeat(LO, 3, axis=0), 3, axis=1)[:h, :w]
    HIp = np.repeat(np.repeat(HI, 3, axis=0), 3, axis=1)[:h, :w]
    sure = (g <= LOp - thr) | (g >= HIp + thr + 1)
    ta, tb = g < HIp - thr, g > LOp + thr + 1
    amb = ~sure & (ta | tb)
    if roi is not None:
        amb &= roi
    if cell_gray is None:
        cell_gray = np.pad(gray, ((0, 3 * ny - h), (0, 3 * nx - w)), mode='edge')
    cg = cell_gray[:3 * ny, :3 * nx].astype(np.int32).reshape(ny, 3, nx, 3)
    dirty = (cg.min(axis=(1, 3)) < HI - thr) | (cg.max(axis=(1, 3)) > LO + thr + 1)
    if roi is not None:
        rp = np.pad(np.asarray(roi, bool), ((0, 3 * ny - h), (0, 3 * nx - w)))
        dirty &= rp.reshape(ny, 3, nx, 3).any(axis=(1, 3))
    code = (C >= 179).sum(0) * 4 + (C >= 263).sum(0)
    return dict(ambiguous=int(amb.sum()), entries=int((amb & ta).sum() + (amb & tb).sum()), centre_counts=C,
                dirty_roi_cells=int(dirty.sum()), codes=np.bincount(code[dirty], minlength=16),
                amb=amb, ta=ta, tb=tb)


def residual_mask_lattice(gray, thr: int, levels, roi=None, stats: Optional[dict] = None, cell_gray=None):
    """numpy twin of the CUDA rank-count stage (csrc/vi_rank.cuh): exact window
    counts only at the centre of every 3x3 cell; |C(p) - C(q)| <= 21 * L1(p, q)
    <= 42 inside a cell, so C(centre) >= 263 proves C >= 221 and C(centre) <= 178
    proves C <= 220 for all nine pixels.  That brackets the median of the whole
    cell between two levels; four thresholds per cell then decide a pixel
    (defect / clean / ambiguous) and ambiguous pixels get an exact rank count.
    Equals residual_mask_direct for ANY level set (tests/test_restate_vs_cv2.py).
    `stats` receives lattice_stats' counts and pivot_counts, the exact window count of every list entry at its
    own pivot."""
    levels = sorted(int(v) for v in levels)
    h, w = gray.shape
    g = gray.astype(np.int32)
    _, LO, HI = _lattice_brackets(gray, thr, levels)
    LOp = np.repeat(np.repeat(LO, 3, axis=0), 3, axis=1)[:h, :w]
    HIp = np.repeat(np.repeat(HI, 3, axis=0), 3, axis=1)[:h, :w]
    sure = (g <= LOp - thr) | (g >= HIp + thr + 1)
    clean = (g >= HIp - thr) & (g <= LOp + thr + 1)
    amb = ~sure & ~clean
    if roi is not None:
        amb &= roi
    out = sure.copy()
    p10 = np.pad(gray, 10, mode='edge')
    st = lattice_stats(gray, thr, levels, roi, cell_gray) if stats is not None else None
    piv = []
    for y, x in zip(*np.nonzero(amb)):
        win = p10[y:y + 21, x:x + 21]
        ca, cb = int((win <= g[y, x] + thr).sum()), int((win <= g[y, x] - thr - 1).sum())
        out[y, x] = ca <= 220 or cb >= 221
        if st is not None:
            piv += ([ca] if st['ta'][y, x] else []) + ([cb] if st['tb'][y, x] else [])
    if stats is not None:
        stats.update({k: v for k, v in st.items() if k not in ('amb', 'ta', 'tb')})
        stats['pivot_counts'] = np.array(piv, np.int32)
    return out


def select_levels(hist, t_apx: int, thr: int, bright: bool = False):
    """The median stage's three levels (csrc/vi_unit.cuh:99-137, select_levels): the lower median m of one
    Otsu class of `hist` split at t_apx (the dark class g <= t_apx, or the bright one), then
    [m - s, m, m + s] clamped to 0..254, s the largest power of two <= max(thr // 3, 1), at most 16.
    An empty class takes m = t_apx."""
    hist = np.asarray(hist, np.int64)
    cum = np.cumsum(hist)
    npix = int(cum[-1])
    nd = int(cum[t_apx])
    nb = npix - nd
    ncls = nb if bright else nd
    tgt = nd + (nb + 1) // 2 if bright else (nd + 1) // 2
    m = int(np.argmax(cum >= tgt)) if ncls else int(t_apx)
    s = 1
    lim = max(thr // 3, 1)
    while s * 2 <= lim and s < 16:
        s *= 2
    return [min(254, max(0, m - s)), min(254, max(0, m)), min(254, max(0, m + s))]


# --------------------------------------------------------------------------- K14/K15
def contour_free_filter(mask, min_area: int, seg_area: int):
    """findContours(EXTERNAL) + contourArea + drawContours(FILLED) + area filter
    (indexing_ui.py:1540-1558) == per 8-component of the 4-bg hole-filled mask H:
    A2 = 2*Q4 + Q3 over 2x2 windows; keep iff 2*min <= A2 <= 2*max
    (SURVEY A.10).  Returns (defect_mask 0/255 or None, n_kept)."""
    H = fill_holes_4bg(mask) > 0
    lab, n = label8(H)
    max_area = max(int(min_area), int(seg_area * 0.98))
    if n == 0:
        return None, 0
    Hi = H.astype(np.int32)
    cnt = Hi[:-1, :-1] + Hi[:-1, 1:] + Hi[1:, :-1] + Hi[1:, 1:]
    # a window with >=3 set pixels lies in one component: take the max label in it
    lw = np.maximum(np.maximum(lab[:-1, :-1], lab[:-1, 1:]), np.maximum(lab[1:, :-1], lab[1:, 1:]))
    q4 = np.bincount(lw[cnt == 4], minlength=n + 1)
    q3 = np.bincount(lw[cnt == 3], minlength=n + 1)
    a2 = 2 * q4 + q3
    keep = (a2 >= 2 * int(min_area)) & (a2 <= 2 * max_area)
    keep[0] = False
    if not keep.any():
        return None, 0
    return (keep[lab] * 255).astype(np.uint8), int(keep.sum())


# --------------------------------------------------------------------------- adaptive threshold
_SMALL_GAUSS_F32 = dict(_SMALL_GAUSS)
_SMALL_GAUSS_F32[9] = [4 / 256, 13 / 256, 30 / 256, 51 / 256, 60 / 256, 51 / 256, 30 / 256, 13 / 256, 4 / 256]


def gaussian_kernel_f32(k: int):
    """cv2.getGaussianKernel(k, 0, CV_32F): the taps of adaptiveThreshold's Gaussian mean
    (OpenCV 4.13 hard-codes the kernels up to 9 taps)."""
    if k in _SMALL_GAUSS_F32:
        return np.array(_SMALL_GAUSS_F32[k], np.float32)
    sigma = ((k - 1) * 0.5 - 1) * 0.3 + 0.8
    s2 = -0.5 / (sigma * sigma)
    kern = np.array([math.exp(s2 * (i - (k - 1) * 0.5) ** 2) for i in range(k)], np.float64)
    return (kern * (1.0 / kern.sum())).astype(np.float32)


def _fma32(a, b, c):
    # float32 fused multiply-add: the float64 product of two float32 is exact; the one extra
    # rounding of the float64 sum can differ from a true FMA only on a double-rounding tie
    return (a.astype(np.float64) * np.float64(b) + c.astype(np.float64)).astype(np.float32)


def adaptive_inv_mask(img, block: int, C: int):
    """cv2.adaptiveThreshold(img, 255, ADAPTIVE_THRESH_GAUSSIAN_C, THRESH_BINARY_INV, bs, C)
    (segmentation.py:83-86; SURVEY A.4): float32 separable Gaussian with BORDER_REPLICATE in the
    operation order of OpenCV's vector path (rows: tap-by-tap FMAs from the first product; columns:
    centre * k[r], then FMAs of (below + above) * k[r+i]), mean rounded half-to-even to uint8,
    255 where img - mean <= -C."""
    bs = max(3, int(block) | 1)
    k = gaussian_kernel_f32(bs)
    r = bs // 2
    h, w = img.shape
    p = np.pad(img, ((0, 0), (r, r)), mode='edge').astype(np.float32)
    s = p[:, 0:w] * k[0]
    for i in range(1, bs):
        s = _fma32(p[:, i:i + w], k[i], s)
    q = np.pad(s, ((r, r), (0, 0)), mode='edge')
    o = q[r:r + h] * k[r]
    for i in range(1, r + 1):
        o = _fma32(q[r + i:r + i + h] + q[r - i:r - i + h], k[r + i], o)
    mean = np.clip(np.rint(o), 0, 255).astype(np.int32)
    return np.where(img.astype(np.int32) - mean <= -int(C), 255, 0).astype(np.uint8)


# --------------------------------------------------------------------------- canny
def canny_edges(gray, low: int, high: int):
    """cv2.Canny(gray, low, high) with aperture 3 and the L1 gradient (indexing_ui.py:1537), integer
    throughout: Sobel with BORDER_REPLICATE, m = |gx| + |gy| (0 outside the crop), non-maximum
    suppression by the 15-bit fixed-point tan 22.5 / tan 67.5 sectors, candidates m > low, strong
    m > high, hysteresis = candidates 8-connected to a strong candidate."""
    if low > high:
        low, high = high, low
    low, high = int(math.floor(low)), int(math.floor(high))
    h, w = gray.shape
    g = np.pad(gray.astype(np.int32), 1, mode='edge')

    def px(dy, dx):
        return g[1 + dy:1 + dy + h, 1 + dx:1 + dx + w]
    gx = (px(-1, 1) + 2 * px(0, 1) + px(1, 1)) - (px(-1, -1) + 2 * px(0, -1) + px(1, -1))
    gy = (px(1, -1) + 2 * px(1, 0) + px(1, 1)) - (px(-1, -1) + 2 * px(-1, 0) + px(-1, 1))
    m = np.abs(gx) + np.abs(gy)
    mp = np.pad(m, 1, mode='constant')

    def mg(dy, dx):
        return mp[1 + dy:1 + dy + h, 1 + dx:1 + dx + w]
    ax = np.abs(gx).astype(np.int64)
    ay15 = np.abs(gy).astype(np.int64) << 15
    tg22x = ax * 13573
    tg67x = tg22x + (ax << 16)
    horiz = ay15 < tg22x
    vert = ~horiz & (ay15 > tg67x)
    diag = ~horiz & ~vert
    same_sign = ~((gx ^ gy) < 0)
    ok_h = (m > mg(0, -1)) & (m >= mg(0, 1))
    ok_v = (m > mg(-1, 0)) & (m >= mg(1, 0))
    ok_d = np.where(same_sign, (m > mg(-1, -1)) & (m > mg(1, 1)), (m > mg(-1, 1)) & (m > mg(1, -1)))
    cand = (m > low) & ((horiz & ok_h) | (vert & ok_v) | (diag & ok_d))
    strong = cand & (m > high)
    lab, n = ndi.label(cand, structure=np.ones((3, 3), np.uint8))
    keep = np.zeros(n + 1, bool)
    keep[np.unique(lab[strong])] = True
    keep[0] = False
    return (keep[lab] * 255).astype(np.uint8)


# --------------------------------------------------------------------------- full unit
def segment_cell(gray, method='otsu', gaussian_blur=3, morph_kernel=3, info: Optional[dict] = None,
                 adapt_block=51, adapt_C=10):
    """segmentation.py:75-100."""
    img = gaussian_blur_u8(gray, gaussian_blur)
    if method == 'adaptive':
        mask = adaptive_inv_mask(img, adapt_block, adapt_C)
    else:
        t, mask = otsu_inv_mask(img)
        if info is not None:
            info['otsu_t'] = t
    mask = morph_close_open(mask, morph_kernel)
    return fill_holes_4bg(mask)


def detect_defects(gray, seg_mask, threshold=24, min_area=20, erode_px=6, levels=None,
                   info: Optional[dict] = None):
    """indexing_ui.py:1486-1560, threshold method, contour-free."""
    seg_bin = ((seg_mask > 0) * 255).astype(np.uint8)
    if erode_px > 0:
        seg_bin = erode_square(seg_bin, int(erode_px))
    lc = largest_component(seg_bin)
    if lc is None:
        return None
    roi = lc[0]
    seg_area = lc[1]
    if info is not None:
        info['roi'] = (roi * 255).astype(np.uint8)
        info['seg_area'] = seg_area
    if levels is None:
        resid = residual_mask_direct(gray, int(threshold))
    else:
        resid = residual_mask_rank(gray, int(threshold), levels, info)
    mask = ((resid & roi) * 255).astype(np.uint8)
    mask = open_cross3(mask)
    out, n_kept = contour_free_filter(mask, int(min_area), seg_area)
    if info is not None:
        info['n_kept'] = n_kept
    return out


# --------------------------------------------------------------------------- frame ingest (SURVEY n3, A.1)
def gray_from_argb32(arr_bgra):
    """Integer restatement of segmentation.py:20-23: OpenCV's 15-bit BGR2GRAY weights meet the reversed channels,
    gray = (R*3735 + G*19235 + B*9798 + 16384) >> 15 with B,G,R the memory order of QImage ARGB32."""
    b = arr_bgra[:, :, 0].astype(np.uint32); g = arr_bgra[:, :, 1].astype(np.uint32); r = arr_bgra[:, :, 2].astype(np.uint32)
    return ((r * 3735 + g * 19235 + b * 9798 + 16384) >> 15).astype(np.uint8)


def gray8_from_gray16(arr_u16):
    """(arr / 256).astype(uint8) on uint16 == the high byte (indexing_ui.py:153-155)."""
    return (arr_u16 >> 8).astype(np.uint8)
