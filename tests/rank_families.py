"""Adversarial inputs for the median residual stage |gray - medianBlur(gray, 21)| > thr (csrc/vi_rank.cuh; its numpy
twin oracle/restate.py: residual_mask_lattice; tests/test_rank_model.py, tests/test_gpu_median_residual.py).

Images: every generator takes a numpy Generator, h, w and thr and returns a uint8 [h][w] crop.  They aim at the places
where a rank count is decided by one pixel: windows that count exactly 220 / 221 at a pivot (period-1 checkerboards,
stripes and checkerboards up to period 21), residuals of exactly thr - 1, thr, thr + 1 (ramps with sparse dots), ties
everywhere (constant crops), pivots past the byte range (0 / 255 crops at thr 0, 1, 254, 255) and cells whose gray
min / max sit exactly on the clean range's ends U2 = HI - thr and U3 = LO + thr + 1 (3x3 blocks).
ROIs: bool [h][w] masks.  Level sets: three sorted levels in 0..255, caller-chosen as the debug entry takes them."""
import cv2
import numpy as np

from oracle import restate as S


def reference(gray, thr, roi):
    """What the stage must give: cv2's median residual inside the ROI."""
    return (cv2.absdiff(gray, cv2.medianBlur(gray, 21)) > thr) & roi


# ----------------------------------------------------------------------------- images
def noise(rng, h, w, thr):
    return rng.integers(0, 256, (h, w), dtype=np.uint8)


def narrow_noise(rng, h, w, thr):
    """noise a few thr wide: most pixels sit near the bracket"""
    c = int(rng.integers(40, 216))
    s = max(2, min(thr, 40))
    return np.clip(c + rng.integers(-s, s + 1, (h, w)), 0, 255).astype(np.uint8)


def constant(rng, h, w, thr):
    return np.full((h, w), int(rng.integers(0, 256)), np.uint8)


def _two_values(rng, thr):
    a = int(rng.integers(0, 256 - thr - 1)) if thr < 255 else 0
    d = [thr, thr + 1, thr + 2, max(thr - 1, 1), int(rng.integers(1, 256))][int(rng.integers(0, 5))]
    return a, min(a + d, 255)


def stripes(rng, h, w, thr):
    p = int(rng.integers(1, 22))
    a, b = _two_values(rng, thr)
    yy, xx = np.mgrid[0:h, 0:w]
    k = xx if rng.random() < 0.5 else yy
    return np.where((k // p) % 2 == 0, a, b).astype(np.uint8)


def checker(rng, h, w, thr):
    p = 1 if rng.random() < 0.5 else int(rng.integers(2, 22))
    a, b = _two_values(rng, thr)
    yy, xx = np.mgrid[0:h, 0:w]
    return np.where(((xx // p) + (yy // p)) % 2 == 0, a, b).astype(np.uint8)


def ramp_dots(rng, h, w, thr):
    """an x, y or diagonal ramp (its median is about the pixel itself) with sparse dots at +-(thr - 1, thr, thr + 1)"""
    yy, xx = np.mgrid[0:h, 0:w]
    sx, sy = [(1.0, 0.0), (0.0, 1.0), (0.37, 0.61)][int(rng.integers(0, 3))]
    span = max(1, 255 - 2 * (thr + 1))
    g = thr + 1 + np.floor((sx * xx + sy * yy) * rng.uniform(0.05, 1.5)).astype(np.int64) % span
    dots = rng.random((h, w)) < 0.06
    d = rng.choice([thr - 1, thr, thr + 1], (h, w)) * rng.choice([-1, 1], (h, w))
    return np.clip(np.where(dots, g + d, g), 0, 255).astype(np.uint8)


def salt_pepper(rng, h, w, thr):
    g = np.full((h, w), int(rng.integers(0, 256)), np.int64)
    u = rng.random((h, w))
    f = rng.uniform(0.02, 0.6)
    g[u < f / 2] = 0
    g[(u >= f / 2) & (u < f)] = 255
    return g.astype(np.uint8)


def extremes(rng, h, w, thr):
    """0 / 255 only: pivots g + thr and g - thr - 1 run past 0..255 (SWAR pivots -1 and >= 255)"""
    return np.where(rng.random((h, w)) < rng.uniform(0.2, 0.8), 0, 255).astype(np.uint8)


def blocks3(rng, h, w, thr, levels=None):
    """3x3 cells of one value each; a third of them moved to HI - thr - 1, HI - thr, LO + thr + 1 or LO + thr + 2
    without crossing a level, so the window counts (and the cells' brackets) stay and their min / max sit exactly on
    an end of the clean range or one past it."""
    ny, nx = (h + 2) // 3, (w + 2) // 3
    c = int(rng.integers(20, 236))
    cells = np.clip(c + rng.integers(-12, 13, (ny, nx)), 0, 255)
    g = np.repeat(np.repeat(cells, 3, 0), 3, 1)[:h, :w].astype(np.uint8)
    lv = sorted(levels if levels is not None else S.select_levels(np.bincount(g.ravel(), minlength=256), c, thr))
    st = {}
    S.residual_mask_lattice(g, thr, lv, stats=st)
    C = st['centre_counts']
    n179, n263 = (C >= 179).sum(0), (C >= 263).sum(0)
    LO = np.array([-1] + lv)[3 - n179]
    HI = np.array(lv + [255])[3 - n263]
    out = np.repeat(np.repeat(cells, 3, 0), 3, 1)
    lva = np.array(lv)
    for j in range(ny):
        for i in range(nx):
            if rng.random() > 0.33:
                continue
            v = cells[j, i]
            for t in rng.permutation([HI[j, i] - thr - 1, HI[j, i] - thr, LO[j, i] + thr + 1, LO[j, i] + thr + 2]):
                if 0 <= t <= 255 and np.array_equal(v <= lva, t <= lva):
                    out[3 * j:3 * j + 3, 3 * i:3 * i + 3] = t
                    break
    return out[:h, :w].astype(np.uint8)


IMAGES = {f.__name__: f for f in (noise, narrow_noise, constant, stripes, checker, ramp_dots, salt_pepper, extremes, blocks3)}
THRS = (0, 1, 2, 7, 24, 60, 127, 254, 255)


# ----------------------------------------------------------------------------- ROIs
def roi_full(rng, h, w):
    return np.ones((h, w), bool)


def roi_empty(rng, h, w):
    return np.zeros((h, w), bool)


def roi_corners(rng, h, w):
    r = np.zeros((h, w), bool)
    r[0, 0] = r[0, -1] = r[-1, 0] = r[-1, -1] = True
    return r


def roi_ring(rng, h, w):
    """the 10 pixels along the crop edge: every window is clipped"""
    r = np.ones((h, w), bool)
    r[10:h - 10, 10:w - 10] = False
    return r


def roi_edge29(rng, h, w):
    """ROI left edge at x = 29..34 (cells that straddle a mask word), or a band that ends there"""
    x0 = int(rng.integers(29, 35))
    r = np.zeros((h, w), bool)
    if rng.random() < 0.5:
        r[:, x0:] = True
    else:
        r[:, :x0 + 1] = True
    return r


def roi_random(rng, h, w):
    return rng.random((h, w)) < 0.5


ROIS = {f.__name__: f for f in (roi_full, roi_empty, roi_corners, roi_ring, roi_edge29, roi_random)}


# ----------------------------------------------------------------------------- level sets
def level_sets(rng, gray, thr):
    """name -> three sorted levels: select_levels' choice, around the true median, all equal, the extremes and far
    from the data (every cell dirty)."""
    hist = np.bincount(gray.ravel(), minlength=256)
    t = int(cv2.threshold(gray.reshape(1, -1), 0, 255, cv2.THRESH_BINARY + cv2.THRESH_OTSU)[0])
    m = int(np.partition(gray.ravel(), (gray.size - 1) // 2)[(gray.size - 1) // 2])
    v = int(rng.integers(0, 256))
    return {
        'select': S.select_levels(hist, t, thr),
        'select_bright': S.select_levels(hist, t, thr, True),
        'median': [max(m - 1, 0), m, min(m + 1, 255)],
        'equal': [v, v, v],
        'zero': [0, 0, 0],
        'top': [254, 254, 254],
        'far': [255, 255, 255] if m < 128 else [0, 0, 0],
    }


def cmm_view(gray, pad):
    """The bytes the kernel's cell min / max pass (vi_rank.cuh: rank_cmm) reads for cell columns 0 .. 3 * nlx - 1:
    the crop row at its pitch with `pad` past w, words past the row's last crop word clamped to it."""
    h, w = gray.shape
    nx = (w + 2) // 3
    nq = (w + 3) // 4
    words = nq + (1 - nq % 2)                  # vi_device.cuh: gray_pitch (odd word count)
    row = np.full((h, 4 * words), pad, np.uint8)
    row[:, :w] = gray
    cols = np.arange(3 * nx)
    b = np.minimum(cols >> 2, nq - 1) * 4 + (cols & 3)
    rows = np.minimum(np.arange(3 * ((h + 2) // 3)), h - 1)          # rows past the crop repeat the last
    return row[rows][:, b]
