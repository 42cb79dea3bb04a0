"""The median residual stage |gray - medianBlur(gray, 21)| > thr inside the ROI (csrc/vi_rank.cuh) against cv2,
pixel by pixel, and its counts against the numpy twin (oracle/restate.py: lattice_stats).

The final defect mask comes after a 3x3-cross opening, which erases a wrong residual bit on any pixel that is not part
of a whole cross: the pixels whose rank count is decided exactly are the ones it hides.  So:
  1. vi_debug_rank_residual runs the stage's device functions alone on caller-chosen levels and returns the raw
     candidate mask and the list counts.  Every case is compared bit for bit with cv2, its entry count with the twin's,
     and it is run again with the dirty-cell and ambiguous-pixel lists capped (ccap, ecap), which sends the same pixels
     through the other paths: a warp per entry (<= 192 entries), a thread per entry (SWAR words or the clipped
     loop), the inline count past ecap, cells classified on the spot past ccap.  The test asserts each path and each
     window geometry (interior, clipped edges and corners, the four byte phases (x - 10) & 3) was taken.
  2. The inspection kernels record n_ambiguous per unit; it must equal the twin's entry count on the unit's ROI with
     the levels the kernel chooses (restate.select_levels at the device's t_apx).

Run on the B200 box: python -m pytest tests/test_gpu_median_residual.py -m gpu"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

from oracle import ref_cv2 as R
from oracle import restate as S
import vi_b200
from vi_b200 import _lib
import rank_families as F
from test_gpu_unit_sequences import assert_sequences, run_device, shelf_layout, sm_count

CCAP, ECAP = 4096, 16384          # vi_rank.cuh: kDirtyListCap, kExactListCap
WARP_MAX = 192                    # vi_rank.cuh: kExactWarpMax


@pytest.fixture(autouse=True)
def opencv_otsu_scan():
    """OpenCV's C++ Otsu scan, which the kernels follow (test_gpu_otsu.py)."""
    ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    yield
    cv2.ipp.setUseIPP(ipp)


@pytest.fixture(scope="module")
def insp():
    i = vi_b200.Inspector(0)
    yield i
    i.close()


def stage(insp, gray, roi, levels, thr, ccap=CCAP, ecap=ECAP, pad=None):
    """vi_debug_rank_residual: (return code, mask bool [h][w], raw words [h][wpr], entries, dirty, otsu_t)."""
    import torch
    h, w = gray.shape
    wpr = (w + 31) // 32
    pad = int(gray[0, -1]) if pad is None else pad
    dg = torch.from_numpy(np.ascontiguousarray(gray)).cuda()
    dr = torch.from_numpy(np.ascontiguousarray(roi).astype(np.uint8) * 255).cuda()
    out = torch.full((h, wpr), -1, dtype=torch.int32, device="cuda")
    lv = (C.c_int * 3)(*levels)
    cnt = (C.c_int * 3)(-1, -1, -1)
    torch.cuda.synchronize()
    rc = insp._lib.vi_debug_rank_residual(insp._ctx, C.c_void_p(dg.data_ptr()), C.c_void_p(dr.data_ptr()), w, h, lv,
                                          thr, ccap, ecap, pad, C.c_void_p(out.data_ptr()), cnt)
    torch.cuda.synchronize()
    words = out.cpu().numpy().view(np.uint32)
    bits = np.unpackbits(words.view(np.uint8).reshape(h, -1), axis=1, bitorder='little').astype(bool)
    return rc, bits[:, :w], bits[:, w:], cnt[0], cnt[1], cnt[2]


class Coverage:
    """Which exact-count paths and window geometries the harness calls took (from the counts and the twin's list)."""

    def __init__(self):
        self.paths = dict(warp=0, thread=0, inline=0, cold=0)
        self.geom = set()

    def add(self, st, gray_shape, entries, dirty, ccap, ecap):
        listed = min(entries, ecap)
        if 0 < listed <= WARP_MAX:
            self.paths['warp'] += 1
        if listed > WARP_MAX:
            self.paths['thread'] += 1
        if entries > ecap:
            self.paths['inline'] += 1
        if dirty > ccap:
            self.paths['cold'] += 1
        if listed == 0:
            return
        h, w = gray_shape
        ys, xs = np.nonzero(st['amb'])
        left, right, top, bot = xs < 10, xs + 10 > w - 1, ys < 10, ys + 10 > h - 1
        inner = ~(left | right | top | bot)
        path = 'thread' if listed > WARP_MAX else 'warp'
        for name, m in (('left', left), ('right', right), ('top', top), ('bottom', bot), ('interior', inner),
                        ('corner', (left | right) & (top | bot))):
            if m.any():
                self.geom.add((path, name))
        if path == 'thread':
            for ph in np.unique((xs[inner] - 10) & 3):
                self.geom.add(('phase', int(ph)))


def check_case(insp, cov, key, gray, roi, lv, thr, caps=False):
    """One input: the mask against cv2 and the counts against the twin for pads = last pixel, 0 and 255; with
    `caps`, every (ccap, ecap) of the sweep gives the same mask and counts."""
    want = F.reference(gray, thr, roi)
    st = S.lattice_stats(gray, thr, lv, roi)
    res = []
    for pad in (None, 0, 255):
        p = int(gray[0, -1]) if pad is None else pad
        rc, mask, tail, ent, dirty, _ = stage(insp, gray, roi, lv, thr, pad=p)
        _lib.check(rc)
        assert np.array_equal(mask, want), (key, pad, int((mask != want).sum()))
        assert not tail.any(), (key, 'padding bits')
        assert ent == st['entries'], (key, pad, ent, st['entries'])
        want_dirty = S.lattice_stats(gray, thr, lv, roi, F.cmm_view(gray, p))['dirty_roi_cells']
        assert dirty == want_dirty, (key, pad, dirty, want_dirty)
        cov.add(st, gray.shape, ent, dirty, CCAP, ECAP)
        res.append((ent, dirty))
    if caps:
        for ccap in (CCAP, 0, 1, 7):
            for ecap in (ECAP, 0, 1, WARP_MAX, WARP_MAX + 1):
                rc, mask, tail, ent, dirty, _ = stage(insp, gray, roi, lv, thr, ccap, ecap)
                _lib.check(rc)
                assert np.array_equal(mask, want), (key, ccap, ecap, int((mask != want).sum()))
                assert (ent, dirty) == res[0], (key, ccap, ecap, ent, dirty, res[0])
                cov.add(st, gray.shape, ent, dirty, ccap, ecap)
    return st


WIDTHS = [1, 2, 3, 4, 5, 20, 21, 22, 31, 32, 33, 34, 77, 78, 79, 80, 96, 97, 316, 1500]
HEIGHTS = [1, 2, 3, 4, 21, 22, 23, 24, 25, 47, 48, 49, 315]


def shapes():
    """Every width with three heights (every height with several widths), the 1500-wide unit whose V pass has 16
    tasks (the Otsu scan runs inside the cell pass), and the thin units at the size bound."""
    out = []
    for i, w in enumerate(WIDTHS):
        for k in range(3):
            h = HEIGHTS[(3 * i + k) % len(HEIGHTS)]
            if w * h <= 316 * 315:
                out.append((h, w))
    return out + [(315, 316), (24, 1500), (49, 1500), (1, 4096), (8192, 1)]


def test_harness_against_cv2_on_every_family_and_cap(insp):
    rng = np.random.default_rng(31)
    cov = Coverage()
    n = 0
    for (h, w) in shapes():
        big = h * w > 60000
        for fi, (name, img) in enumerate(F.IMAGES.items()):
            if big and fi % 3:
                continue
            thr = int(rng.choice(F.THRS))
            g = img(rng, h, w, thr)
            lsets = F.level_sets(rng, g, thr)
            rnames = list(F.ROIS)
            for li, lname in enumerate(['select', list(lsets)[1 + (fi + h) % (len(lsets) - 1)]]):
                rname = rnames[(fi + li + w) % len(rnames)]
                roi = F.ROIS[rname](rng, h, w)
                caps = (not big) and (fi + li + h + w) % 4 == 0
                check_case(insp, cov, (h, w, name, thr, lname, rname), g, roi, sorted(lsets[lname]), thr, caps)
                n += 1
    # dense ambiguous lists at every cap: noise at a low threshold on a full ROI and on the ring
    for (h, w) in [(48, 97), (25, 80), (315, 316)]:
        for thr, rname in [(2, 'roi_full'), (7, 'roi_ring'), (0, 'roi_random')]:
            g = F.noise(rng, h, w, thr)
            lv = sorted(F.level_sets(rng, g, thr)['select'])
            check_case(insp, cov, (h, w, 'noise', thr, 'select', rname), g, F.ROIS[rname](rng, h, w), lv, thr, True)
            n += 1
    print(f"\n[rank] {n} inputs; paths {cov.paths}; geometry {sorted(cov.geom, key=str)}")
    assert all(v > 0 for v in cov.paths.values()), cov.paths
    for path in ('warp', 'thread'):
        for name in ('left', 'right', 'top', 'bottom', 'interior', 'corner'):
            assert (path, name) in cov.geom, (path, name)
    assert {('phase', p) for p in range(4)} <= cov.geom


def test_harness_otsu_on_both_placements(insp):
    """otsu_t of the harness is cv2's Otsu threshold of the crop, beside the V pass (narrow) and inside it (1500 px)."""
    rng = np.random.default_rng(8)
    for (h, w) in [(40, 60), (24, 1500), (1, 4096)]:
        g = np.where(rng.random((h, w)) < 0.4, rng.integers(40, 90, (h, w)), rng.integers(150, 230, (h, w))).astype(np.uint8)
        rc, _, _, _, _, t = stage(insp, g, np.ones((h, w), bool), [100, 110, 120], 24)
        _lib.check(rc)
        assert t == int(cv2.threshold(g, 0, 255, cv2.THRESH_BINARY_INV + cv2.THRESH_OTSU)[0]), (h, w)


def test_harness_rejects_bad_arguments(insp):
    g = np.zeros((8, 8), np.uint8)
    r = np.ones((8, 8), bool)
    for kw in (dict(levels=[3, 2, 4]), dict(levels=[0, 0, 256]), dict(levels=[-1, 0, 0]), dict(thr=256), dict(thr=-1),
               dict(ccap=CCAP + 1), dict(ecap=ECAP + 1), dict(ecap=-1), dict(pad=256)):
        a = dict(levels=[1, 2, 3], thr=5, ccap=CCAP, ecap=ECAP, pad=0)
        a.update(kw)
        rc = stage(insp, g, r, a['levels'], a['thr'], a['ccap'], a['ecap'], a['pad'])[0]
        assert rc == _lib.VI_ERR_ARG, kw
    import torch
    d = torch.zeros(16, dtype=torch.uint8, device="cuda")
    cnt = (C.c_int * 3)()
    lv = (C.c_int * 3)(1, 2, 3)
    for w, h in ((0, 4), (4097, 1), (1, 8193), (4096, 4097)):
        assert insp._lib.vi_debug_rank_residual(insp._ctx, C.c_void_p(d.data_ptr()), C.c_void_p(d.data_ptr()), w, h, lv,
                                                5, CCAP, ECAP, 0, C.c_void_p(d.data_ptr()), cnt) == _lib.VI_ERR_ARG


# ---- 2. the inspection kernels: n_ambiguous per unit ------------------------------------------------------------------

# (w, h, noise sigma, x0 & 15): plates whose noise is strong against the threshold, mixed with quiet ones
UNITS = [(316, 315, 14, 3), (96, 96, 0, 5), (150, 141, 9, 1), (40, 33, 3, 7), (200, 150, 20, 0), (97, 111, 1, 2),
         (64, 64, 6, 4), (250, 60, 12, 6), (20, 300, 4, 14)]


def noisy_frames(boxes, sig, n, H, W, seed0):
    from vi_b200 import synth
    out = []
    for i in range(n):
        rng = np.random.default_rng(seed0 + i)
        f = synth.make_frame(seed0 + i, [b for b, _ in boxes], H=H, W=W, inset=5, jitter=2).astype(np.float64)
        for ((x, y, w, h), _), s in zip(boxes, sig):
            f[y:y + h, x:x + w] += rng.normal(0, s, (h, w))
        out.append(np.clip(np.rint(f), 0, 255).astype(np.uint8))
    return np.stack(out)


def device_tapx(insp, hists):
    import torch
    H = np.ascontiguousarray(hists, np.int64)
    dh = torch.from_numpy(H.astype(np.uint32).view(np.int32)).cuda()
    dn = torch.from_numpy(H.sum(1).astype(np.int32)).cuda()
    out = torch.empty((len(H), 3), dtype=torch.int32, device="cuda")
    _lib.check(insp._lib.vi_debug_otsu(insp._ctx, C.c_void_p(dh.data_ptr()), C.c_void_p(dn.data_ptr()), len(H),
                                       C.c_void_p(out.data_ptr())))
    torch.cuda.synchronize()
    return out.cpu().numpy()[:, 1]


KERNELS = {'spec': dict(), 'general': dict(gaussian_blur=5, morph_kernel=5), 'arena': dict()}


@pytest.mark.parametrize("kname", list(KERNELS))
def test_kernels_record_the_twin_entry_count(insp, kname):
    """Masks and records against the cv2 oracle, and per unit n_ambiguous == the twin's entries with the kernel's
    levels (select_levels at t_apx of the blurred crop's histogram) and the oracle's ROI.  The grid mixes units of
    <= 192, > 192 and > 16,384 entries and of > 4,096 dirty ROI cells in the same CTAs."""
    import torch
    from vi_b200.grid import Grid
    kw = dict(KERNELS[kname], threshold=6)
    units = UNITS + ([(640, 480, 10, 0)] if kname == 'arena' else [])
    boxes, right, bottom = shelf_layout([(w, h, ph) for w, h, _, ph in units], 1008)
    sms = sm_count()
    n = max(2, -(-4 * sms // len(units)))
    frames = noisy_frames(boxes, [s for _, _, s, _ in units], n, bottom + 8, 1024, 500)
    assert_sequences([(w, h) for w, h, _, _ in units], n, sms)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    rec, seg, dfm = run_device(insp, torch.from_numpy(frames).cuda(), vi_b200.default_params(**kw))
    rp = R.Params(**kw)
    k = kw.get('gaussian_blur', 3)
    buckets = dict(warp=0, thread=0, inline=0, cold=0)
    crops, rois = [], []
    for fi in range(n):
        recs, osegs, odefs = R.inspect_frame(frames[fi], boxes, rp, (), None, True)
        defs = insp.split_masks(dfm[fi])
        segs = insp.split_masks(seg[fi])
        for u, o in enumerate(recs):
            assert np.array_equal(segs[u], osegs[u]), (kname, fi, u, 'seg')
            want = odefs[u] if odefs[u] is not None else np.zeros_like(defs[u])
            assert np.array_equal(defs[u], want), (kname, fi, u, 'defect')
            for f in ('seg_area', 'roi_area', 'defect_area', 'n_kept', 'status'):
                assert rec[fi, u][f] == o[f], (kname, fi, u, f)
            (x, y, w, h), _ = boxes[u]
            crop = np.ascontiguousarray(frames[fi, y:y + h, x:x + w])
            info = {}
            R.detect_defects(crop, osegs[u], 'threshold', rp.threshold, rp.min_area, rp.erode_px, info)
            crops.append((fi, u, crop))
            rois.append(info['roi'] > 0 if info.get('roi') is not None else None)
    hists = [np.bincount(cv2.GaussianBlur(c, (k, k), 0).ravel(), minlength=256) for _, _, c in crops]
    tapx = device_tapx(insp, np.stack(hists))
    for (fi, u, crop), roi, hist, ta in zip(crops, rois, hists, tapx):
        r = rec[fi, u]
        if roi is None or not roi.any():
            assert r['n_ambiguous'] == 0, (kname, fi, u)
            continue
        st = S.lattice_stats(crop, rp.threshold, S.select_levels(hist, int(ta), rp.threshold), roi)
        assert r['n_ambiguous'] == st['entries'], (kname, fi, u, int(r['n_ambiguous']), st['entries'])
        e = st['entries']
        buckets['warp'] += 0 < e <= WARP_MAX
        buckets['thread'] += e > WARP_MAX
        buckets['inline'] += e > ECAP
        buckets['cold'] += st['dirty_roi_cells'] > CCAP
    print(f"\n[rank {kname}] units by path: {buckets}")
    assert all(v > 0 for v in buckets.values()), buckets
