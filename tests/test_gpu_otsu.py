"""The device Otsu threshold against OpenCV's C++ scan (oracle/restate.py: otsu_from_hist, otsu_from_hists) on
adversarial histograms (tests/otsu_families.py), through each place the exact scan runs.

The kernels compute the threshold in two steps (vi_pipeline.cuh): otsu_approx_warp finds the bound `last` from
float32 variances, and otsu_scan runs the reference's double recurrence up to it.  Where the scan runs:
  * on its own warp beside the median stage's cell pass when the V pass has at most 15 tasks (vi_rank.cuh:
    rank_vplan, rank_otsu_aside): every unit narrower than about 1,420 px, e.g. 96 x 96 (8 tasks), 400 x 60 (15),
    500 x 60 (12);
  * inside the cell pass, on the warp kOtsuWarp after its columns, when the V pass has 16 or more tasks: units wider
    than about 1,420 px, e.g. 1500 x 24 (16 chunks of 32 cell slots);
  * after the barrier, on kOtsuWarp alone, without the lattice (defect_method='canny');
  * in the arena kernel (a 640 x 480 unit in the grid puts the whole grid there).

Run on the B200 box: python -m pytest tests/test_gpu_otsu.py -m gpu"""
import ctypes as C
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

from oracle import ref_cv2 as R
from oracle import restate as S
import vi_b200
from vi_b200 import _lib
import otsu_families as F
from test_gpu_unit_sequences import check_oracle, configure, run_bound, run_device, shelf_layout

RAW = dict(gaussian_blur=0, morph_kernel=0)        # a unit's histogram is its pixel multiset


@pytest.fixture(autouse=True)
def opencv_otsu_scan():
    """OpenCV's C++ scan, which the kernels follow: the IPP routine the cv2 wheel dispatches to by default breaks
    exact ties differently (test_gpu_parity.py: test_otsu_threshold_near_ties)."""
    ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    yield
    cv2.ipp.setUseIPP(ipp)


@pytest.fixture
def insp():
    i = vi_b200.Inspector(0)
    yield i
    i.close()


def cv2_otsu(im):
    return int(cv2.threshold(im, 0, 255, cv2.THRESH_BINARY_INV + cv2.THRESH_OTSU)[0])


def device_otsu(insp, H, npix=None):
    """vi_debug_otsu on the rows of H: (return code, [n, 3] = t, t_apx, last)."""
    import torch
    H = np.ascontiguousarray(H, dtype=np.int64)
    npix = H.sum(1) if npix is None else np.asarray(npix)
    dh = torch.from_numpy(H.astype(np.uint32).view(np.int32)).cuda()
    dn = torch.from_numpy(npix.astype(np.int32)).cuda()
    out = torch.full((len(H), 3), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    rc = insp._lib.vi_debug_otsu(insp._ctx, C.c_void_p(dh.data_ptr()), C.c_void_p(dn.data_ptr()), len(H),
                                 C.c_void_p(out.data_ptr()))
    torch.cuda.synchronize()
    return rc, out.cpu().numpy()


# ---- 1. the device functions on about 10^6 histograms ---------------------------------------------------------------

def test_device_otsu_on_a_million_adversarial_histograms(insp):
    """Every family, with pixel counts over 1..2^24 (dense around 2^23 and at 2^24): t equals the reference's
    threshold and the bound `last` is at or after it."""
    rng = np.random.default_rng(2024)
    t0 = time.perf_counter()
    total = 0
    for chunk in range(10):
        H, names = F.mixed(rng, 10000)
        ref = S.otsu_from_hists(H)
        rc, out = device_otsu(insp, H)
        _lib.check(rc)
        t, tapx, last = out.T
        bad = np.nonzero(t != ref)[0]
        assert bad.size == 0, (names[bad[0]], H[bad[0]].sum(), np.nonzero(H[bad[0]])[0], t[bad[0]], ref[bad[0]])
        assert (last >= ref).all() and (last <= 255).all()
        assert ((tapx >= 0) & (tapx <= 255)).all()
        total += len(H)
    print(f"\n[otsu] {total} histograms checked in {time.perf_counter() - t0:.1f} s")


@pytest.mark.parametrize("wh", [(4096, 2049), (4096, 3000), (4096, 4096), (2048, 8192), (4096, 2048), (2048, 2048)])
def test_device_otsu_at_large_unit_sizes(insp, wh):
    """The lone-pixel families at the pixel counts of large units, where a class of one pixel is below FLT_EPSILON
    of the unit (above 2^23) or not (2^23 and below)."""
    n = wh[0] * wh[1]
    rng = np.random.default_rng(n % 997)
    H = np.concatenate([F.trigger(rng, 2000, n), F.trigger_mirror(rng, 2000, n), F.lone_pixels(rng, 2000, n),
                        F.two_spikes(rng, 500, n), F.bimodal(rng, 500, n)])
    ref = S.otsu_from_hists(H)
    rc, out = device_otsu(insp, H)
    _lib.check(rc)
    assert np.array_equal(out[:, 0], ref) and (out[:, 2] >= ref).all()


def test_device_otsu_against_opencv(insp):
    """A sample of every family as images, thresholded by cv2 (IPP off), up to 2^24 pixels."""
    rng = np.random.default_rng(77)
    hs = []
    for f in F.FAMILIES.values():
        for n in (16, 300, 5000, 70000, (1 << 23) + 1, 1 << 24):
            hs.append(f(rng, 2, n))
    H = np.concatenate(hs)
    rc, out = device_otsu(insp, H)
    _lib.check(rc)
    for j, h in enumerate(H):
        im = F.image_of(h, rng)
        assert out[j, 0] == cv2_otsu(im) == S.otsu_from_hist(h), (j, h.sum(), np.nonzero(h)[0])


def test_device_otsu_argument_checks(insp):
    """npix outside 1..2^24, or not its histogram's sum: VI_ERR_ARG, -1 in that row, the other rows computed."""
    h = np.zeros((5, 256), np.int64)
    h[:, 10], h[:, 200] = 3, 5
    h[3, 0] = (1 << 24) + 1 - 8                  # a sum of 2^24 + 1
    h[4] = 0
    npix = np.array([8, 9, 8, (1 << 24) + 1, 0])
    rc, out = device_otsu(insp, h, npix)
    assert rc == _lib.VI_ERR_ARG
    assert (out[[1, 3, 4]] == -1).all()
    assert out[0, 0] == out[2, 0] == S.otsu_from_hist(h[0]) == 10
    assert insp._lib.vi_debug_otsu(insp._ctx, None, None, 0, None) == _lib.VI_OK
    assert insp._lib.vi_debug_otsu(insp._ctx, None, None, 3, None) == _lib.VI_ERR_ARG


# ---- 2. designed histograms through the batch kernels ----------------------------------------------------------------

def rank_tasks(w, h, warps=16, cell=3, vpad=3):
    """rank_vplan(g).ntask (vi_rank.cuh): the scan runs on its own warp when this is <= warps - 1."""
    nslot, nly = (w + cell - 1) // cell + 2 * vpad, (h + cell - 1) // cell
    nchunk = (nslot + 31) >> 5
    nseg = max(1, min(min(4, (warps - 1) // nchunk), (nly + 7) >> 3))
    seg_rows = (((nly + nseg - 1) // nseg) + 7) & ~7
    return nchunk * ((nly + seg_rows - 1) // seg_rows)


def designed_grid(rng, n_small, wide, big=None):
    """n_small units of 4..120 x 4..40 px (at least 16 px), the `wide` (w, h) units in their place and optionally
    one `big` (w, h), on shelves."""
    units = [(int(rng.integers(4, 121)), int(rng.integers(4, 41)), 0) for _ in range(n_small)]
    units = [(w, max(h, (16 + w - 1) // w), p) for w, h, p in units]            # at least 16 px each
    pos = rng.choice(n_small, len(wide), replace=False)
    for k, p in enumerate(sorted(pos)):
        units[p] = (*wide[k], 0)
    if big is not None:
        units.insert(n_small // 2, (*big, 0))
    boxes, right, bottom = shelf_layout(units, 2040, gap=2)
    return boxes, bottom + 4


def designed_frames(boxes, H, n_frames, seed):
    """Frames whose units are random permutations of designed pixel multisets (families in turn), and the
    histograms [frame][unit]."""
    rng = np.random.default_rng(seed)
    fams = list(F.FAMILIES.values())
    frames = np.zeros((n_frames, H, 2048), np.uint8)
    hists = []
    for fi in range(n_frames):
        hs = []
        for u, ((x, y, w, h), _) in enumerate(boxes):
            f = fams[(u + fi) % len(fams)]
            hist = f(rng, 1, w * h)[0]
            frames[fi, y:y + h, x:x + w] = F.image_of(hist, rng, (h, w))
            hs.append(hist)
        hists.append(np.array(hs))
    return frames, hists


def run_designed(insp, boxes, frames, hists, kw):
    import torch
    refc = configure(insp, frames, boxes, kw)
    rec, seg, dfm = run_device(insp, torch.from_numpy(frames).cuda(), vi_b200.default_params(**kw))
    check_oracle(insp, frames, boxes, kw, refc, rec, seg, dfm)
    for fi, hs in enumerate(hists):
        assert np.array_equal(rec['otsu_t'][fi], S.otsu_from_hists(hs)), fi


WIDE = [(1500, 24), (1500, 40), (1440, 30), (400, 60), (500, 60)]


def test_designed_units_scan_aside_and_in_the_cell_pass(insp):
    """1,600 ragged units, blur and morphology off (the general kernel with the median stage's lattice): the small
    ones and 400 x 60 / 500 x 60 scan on their own warp, 1500 x 24, 1500 x 40 and 1440 x 30 inside the cell pass."""
    assert [rank_tasks(w, h) for w, h in WIDE] == [16, 16, 16, 15, 12]
    assert max(rank_tasks(w, h) for w in range(4, 121) for h in range(4, 41)) <= 15
    rng = np.random.default_rng(5)
    boxes, H = designed_grid(rng, 1600, WIDE)
    frames, hists = designed_frames(boxes, H, 2, 31)
    run_designed(insp, boxes, frames, hists, RAW)


def test_designed_units_without_the_lattice(insp):
    """The same kind of grid with Canny defects: no median stage, the scan runs on kOtsuWarp after the barrier."""
    rng = np.random.default_rng(6)
    boxes, H = designed_grid(rng, 1200, WIDE[:2])
    frames, hists = designed_frames(boxes, H, 2, 32)
    run_designed(insp, boxes, frames, hists, dict(RAW, defect_method='canny', threshold=24))


def test_designed_units_in_the_arena_kernel(insp):
    """A 640 x 480 designed unit among 1,200 small ones: the whole grid runs on the arena kernel."""
    rng = np.random.default_rng(7)
    boxes, H = designed_grid(rng, 1200, WIDE[:1], big=(640, 480))
    frames, hists = designed_frames(boxes, H, 2, 33)
    run_designed(insp, boxes, frames, hists, RAW)


# ---- 3. the default kernel on flat patches --------------------------------------------------------------------------------

def flat_frames(boxes, H, n_frames, seed):
    """Units of two or three flat levels (0 and 255 among them), some with a lone dead pixel (0 or 255)."""
    rng = np.random.default_rng(seed)
    frames = np.zeros((n_frames, H, 2048), np.uint8)
    levels = np.array([0, 1, 2, 40, 100, 127, 128, 200, 253, 254, 255])
    for fi in range(n_frames):
        for (x, y, w, h), _ in boxes:
            lv = rng.choice(levels, rng.integers(2, 4), replace=False)
            u = np.full((h, w), lv[0], np.uint8)
            for v in lv[1:]:
                x0, y0 = rng.integers(0, w), rng.integers(0, h)
                u[y0:y0 + rng.integers(1, h + 1), x0:x0 + rng.integers(1, w + 1)] = v
            if rng.random() < 0.5:
                u[rng.integers(0, h), rng.integers(0, w)] = rng.choice([0, 255])
            frames[fi, y:y + h, x:x + w] = u
    return frames


def test_default_kernel_on_flat_patches(insp):
    """Default parameters (3 x 3 blur, the default kernel): otsu_t against cv2 on the blurred crop, masks and
    records against the oracle."""
    import torch
    rng = np.random.default_rng(8)
    units = [(int(rng.integers(3, 160)), int(rng.integers(3, 160)), 0) for _ in range(600)]
    boxes, right, bottom = shelf_layout(units, 2040, gap=2)
    frames = flat_frames(boxes, bottom + 4, 2, 34)
    refc = configure(insp, frames, boxes, {})
    rec, seg, dfm = run_device(insp, torch.from_numpy(frames).cuda(), vi_b200.default_params())
    check_oracle(insp, frames, boxes, {}, refc, rec, seg, dfm)


# ---- 4. units above 2^23 pixels, end to end -------------------------------------------------------------------------------

# (x0, a, gap, m): 1 pixel at x0, m at a, the rest at a + gap.  Above 2^23 pixels the reference skips the lone
# pixel's split; a bound that scored it stops the scan before a and the threshold comes out 0.
TRIGGERS = [(0, 200, 1, 30000), (0, 60, 1, 1000)]


def trigger_frame(w, h, design, mirror=False, seed=0):
    """A (h + 16) x W frame with the unit at (0, 8): the rest level as background, the m pixels as a block of
    rows, the lone pixel apart from it."""
    x0, a, gap, m = design
    lv = (lambda v: 255 - v) if mirror else (lambda v: v)
    fr = np.full((h + 16, max(w, 64)), lv(a + gap), np.uint8)
    u = fr[8:8 + h, :w]
    flat = u.reshape(-1)
    start = (h // 3) * w + w // 4
    flat[start:start + m] = lv(a)
    u[h - 5, w - 7] = lv(x0)
    hist = np.bincount(u.ravel(), minlength=256)
    assert hist.sum() == w * h and hist[lv(x0)] == 1 and hist[lv(a)] == m
    return fr


def run_large(w, h, frames, kw=RAW):
    box = (0, 8, w, h)
    recs, rec = run_bound([(box, 0)], frames, kw)
    for fi in range(len(frames)):
        crop = np.ascontiguousarray(frames[fi, 8:8 + h, :w])
        if kw is RAW:
            assert rec['otsu_t'][fi, 0] == S.otsu_from_hist(np.bincount(crop.ravel(), minlength=256)), fi
    return rec


def check_segment_cell(frame, w, h, kw=RAW):
    insp = vi_b200.Inspector(0)
    try:
        crop = np.ascontiguousarray(frame[8:8 + h, :w])
        got, t = insp.segment_cell(crop, vi_b200.default_params(**kw), return_threshold=True)
        assert t == cv2_otsu(crop if kw is RAW else cv2.GaussianBlur(crop, (3, 3), 0))
        assert np.array_equal(got, R.segment_cell(crop, **kw))
        return t
    finally:
        insp.close()


@pytest.mark.parametrize("wh", [(4096, 2049), (4096, 3000), (4096, 4096), (2048, 8192)])
def test_lone_dark_pixel_above_2_23_pixels(wh):
    """The trigger histograms at 4096 x 2049 (2^23 + 4096 px) and up: the batch call against the oracle (records
    and both masks) and segment_cell's threshold against cv2."""
    w, h = wh
    frames = np.stack([trigger_frame(w, h, d) for d in TRIGGERS])
    rec = run_large(w, h, frames)
    assert list(rec['otsu_t'][:, 0]) == [200, 60]
    assert check_segment_cell(frames[0], w, h) == 200


def test_controls_at_and_above_2_23_pixels():
    """4096 x 2048 (exactly 2^23: the lone pixel's split counts and the reference's threshold is 0), the mirrored
    trigger at 4096 x 4096 (the lone pixel at the bright end) and a default-blur unit with a dead pixel."""
    frames = np.stack([trigger_frame(4096, 2048, d) for d in TRIGGERS])
    rec = run_large(4096, 2048, frames)
    assert list(rec['otsu_t'][:, 0]) == [0, 0]
    frames = np.stack([trigger_frame(4096, 4096, d, mirror=True) for d in TRIGGERS])
    run_large(4096, 4096, frames)
    assert check_segment_cell(frames[0], 4096, 4096) == S.otsu_from_hist(np.bincount(frames[0, 8:4104].ravel(), minlength=256))
    fr = np.full((4112, 4096), 180, np.uint8)
    fr[8 + 1200:8 + 2900, 1000:3100] = 60
    fr[8 + 3000, 3500] = 0
    frames = np.stack([fr, np.where(fr == 180, 250, fr).astype(np.uint8)])
    run_large(4096, 4096, frames, {})
    check_segment_cell(frames[0], 4096, 4096, {})
