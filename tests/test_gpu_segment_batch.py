"""The segmentation-only batch calls (vi_segment_batch, vi_segment_batch_host, Inspector.segment_batch /
segment_batch_host, segmentation.segment_batch) against the cv2 oracle and against vi_inspect_batch on the same frames,
on every kernel that runs them: the segmentation instantiation of the default configuration (tensor boxes, row copies,
a strided view), the general kernel and the arena kernel.

Every unit is compared with oracle/ref_cv2.segment_unit: the mask bit for bit, cx / cy bit for bit, dx, dy, seg_area
and otsu_t (OpenCV's C++ Otsu scan).  It is also compared with vi_inspect_batch's seg outputs: byte masks, seg_stats,
packed seg bits and the record fields the two calls share (n_runs is a diagnostic and is not compared).

Run on the B200 box: python -m pytest tests/test_gpu_segment_batch.py -m gpu"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

from oracle import ref_cv2 as R
import vi_b200
from vi_b200 import synth
from vi_b200.grid import Grid, ref_centroids_from_records
from test_gpu_unit_sequences import (ARENA_UNITS, EXCL, G1, G2, assert_sequences, blur_k, frames_for, make_frames,
                                     shelf_layout, sm_count)

import otsu_families as F

SHARED = ('image', 'unit', 'otsu_t', 'seg_area', 'dx', 'dy', 'cx', 'cy')
SENT = 0xA5


@pytest.fixture(autouse=True)
def opencv_otsu_scan():
    """OpenCV's C++ Otsu scan, which the kernels follow (test_gpu_unit_sequences.py: opencv_otsu_scan)."""
    ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    yield
    cv2.ipp.setUseIPP(ipp)


@pytest.fixture
def insp():
    i = vi_b200.Inspector(0)
    yield i
    i.close()


def outs(insp, n):
    import torch
    return dict(seg_stats=torch.full((n * insp.n_units, 3), -7, dtype=torch.int64, device="cuda"),
                seg_bits=torch.full((n * insp.packed_bytes,), SENT, dtype=torch.uint8, device="cuda"))


def host(o):
    return {k: v.cpu().numpy() for k, v in o.items()}


def segment(insp, ft, p, prof=None, **kw):
    import torch
    if prof is not None:
        vi_b200._lib.check(insp._lib.vi_debug_set_profile(insp._ctx, C.c_void_p(prof.data_ptr())))
    try:
        rec, seg = insp.segment_batch(ft, p, **kw)
        torch.cuda.synchronize()
    finally:
        if prof is not None:
            vi_b200._lib.check(insp._lib.vi_debug_set_profile(insp._ctx, None))
    n = ft.shape[0]
    return rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(n, insp.n_units), seg.cpu().numpy().reshape(n, -1)


def inspect(insp, ft, p, **kw):
    import torch
    rec, seg, _ = insp.inspect_batch(ft, p, **kw)
    torch.cuda.synchronize()
    n = ft.shape[0]
    return rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(n, insp.n_units), seg.cpu().numpy().reshape(n, -1)


def check_against_oracle(insp, frames, boxes, kw, rec, seg, excl=(), refc=None, is_reference=False):
    rp = R.Params(**kw)
    k = blur_k(kw)
    refc = refc or {}
    for fi in range(len(frames)):
        segs = insp.split_masks(seg[fi])
        for u, ((x, y, w, h), _) in enumerate(boxes):
            crop = np.ascontiguousarray(frames[fi, y:y + h, x:x + w])
            mask, c1, dx, dy = R.segment_unit(crop, rp, excl, refc.get(u), is_reference)
            r = rec[fi, u]
            assert r['image'] == fi and r['unit'] == u and r['status'] == vi_b200.STATUS_SEGMENTED
            assert np.array_equal(segs[u], mask), (kw, fi, u, int((segs[u] != mask).sum()))
            assert (r['seg_area'], r['dx'], r['dy']) == (int((mask > 0).sum()), dx, dy), (kw, fi, u)
            c = (c1 if c1 is not None else (float('nan'), float('nan')))
            assert np.float64([r['cx'], r['cy']]).tobytes() == np.float64(c).tobytes(), (kw, fi, u, 'centroid')
            for f in ('roi_area', 'defect_area', 'n_kept', 'n_ambiguous'):
                assert r[f] == 0, (fi, u, f)
            if kw.get('seg_method', 'otsu') != 'adaptive':
                assert r['otsu_t'] == R.otsu_threshold(cv2.GaussianBlur(crop, (k, k), 0) if k else crop), (kw, fi, u)


def check_against_inspect(insp, ft, p, rec, seg, o):
    """vi_inspect_batch on the same frames: the seg outputs and the shared record fields are equal."""
    n = ft.shape[0]
    o2 = outs(insp, n)
    rec2, seg2 = inspect(insp, ft, p, **o2)
    assert np.array_equal(seg, seg2)
    for f in SHARED:
        assert rec[f].tobytes() == rec2[f].tobytes(), f
    for k2, v in host(o2).items():
        assert np.array_equal(o[k2], v), k2


def full_check(insp, frames, boxes, kw, ft=None, excl=(), refc=None, is_reference=False, prof=None):
    import torch
    p = vi_b200.default_params(**kw)
    ft = torch.from_numpy(frames).cuda() if ft is None else ft
    o = outs(insp, frames.shape[0])
    rec, seg = segment(insp, ft, p, prof=prof, **o)
    o = host(o)
    check_against_oracle(insp, frames, boxes, kw, rec, seg, excl, refc, is_reference)
    check_against_inspect(insp, ft, p, rec, seg, o)
    return rec, seg


# ---- 1. the segmentation instantiation of the default configuration ---------------------------------------------------

def seg_profile(insp, n):
    import torch
    return torch.zeros((n * insp.n_units, 48), dtype=torch.int64, device="cuda")


@pytest.mark.parametrize("grid", ["G1", "G2"])
def test_seg_kernel_over_ragged_sequences(insp, grid):
    """G1 (tensor boxes) and G2 (row copies), default parameters, every CTA running at least 3 units.  The phase
    profile is written, which only the segmentation kernel does in this mode."""
    units = G1 if grid == "G1" else G2
    sms = sm_count()
    n = frames_for(len(units), sms)
    assert_sequences([(w, h) for w, h, _ in units], n, sms)
    boxes, _, bottom = shelf_layout(units, 1008)
    frames = make_frames(boxes, n, bottom + 8, 1024, 2000 if grid == "G1" else 2100)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    prof = seg_profile(insp, n)
    full_check(insp, frames, boxes, {}, prof=prof)
    assert int(prof.count_nonzero()) > 0


def test_seg_kernel_on_a_strided_view(insp):
    import torch
    boxes, right, bottom = shelf_layout(G1, 1008)
    n, H, W = 12, bottom + 8, 1024
    frames = make_frames(boxes, n, H, W, 2200)
    big = torch.zeros((n, H + 32, W + 64), dtype=torch.uint8, device="cuda")
    big[:, :H, :W] = torch.from_numpy(frames).cuda()
    view = big[:, :H, :W]
    insp.configure(Grid(boxes=boxes), is_reference=True)
    prof = seg_profile(insp, n)
    full_check(insp, frames, boxes, {}, ft=view, prof=prof)
    assert int(prof.count_nonzero()) > 0


# ---- 2. exclusions, shift and the reference centroids -----------------------------------------------------------------

def test_exclusions_shift_and_ref_centroids(insp):
    """BASELINE configs[3]'s setup: rect + circle exclusions.  The reference image's centroids come from
    segment_batch itself (ref_centroids_from_records), equal the full call's cx / cy, and drive the shift of the others."""
    import torch
    boxes, _, bottom = shelf_layout(G1, 1008)
    n = 10
    frames = make_frames(boxes, n, bottom + 8, 1024, 2300, max_discs=6)
    insp.configure(Grid(boxes=boxes, exclusions=EXCL), is_reference=True)
    ft0 = torch.from_numpy(frames[:1]).cuda()
    rec0, _ = full_check(insp, frames[:1], boxes, {}, excl=EXCL, is_reference=True)
    refc = ref_centroids_from_records(rec0)
    full0, _ = inspect(insp, ft0, vi_b200.default_params())
    assert refc == {u: (float(r['cx']), float(r['cy'])) for u, r in enumerate(full0[0]) if r['cx'] == r['cx']}
    assert refc == {u: c for u, c in ((u, R.segment_unit(np.ascontiguousarray(frames[0, y:y + h, x:x + w]), R.Params(),
                                                         EXCL, None, True)[1]) for u, ((x, y, w, h), _) in enumerate(boxes))
                    if c is not None}
    insp.configure(Grid(boxes=boxes, exclusions=EXCL, ref_centroids=refc), is_reference=False)
    rec, _ = full_check(insp, frames, boxes, {}, excl=EXCL, refc=refc)
    assert (rec['dx'] != 0).any() or (rec['dy'] != 0).any()
    insp.configure(Grid(boxes=boxes, exclusions=EXCL, ref_centroids=refc), is_reference=True)
    rec, _ = full_check(insp, frames, boxes, {}, excl=EXCL, refc=refc, is_reference=True)
    assert (rec['dx'] == 0).all() and (rec['dy'] == 0).all()


# ---- 3. the Otsu scan without a median stage beside it ---------------------------------------------------------------

def designed_units(H, side):
    """One side x side unit per histogram, its pixels the histogram's multiset; blur and morphology off, so the
    unit's Otsu histogram is that multiset.  Returns (boxes, frame)."""
    k = H.shape[0]
    per_row = 1024 // (side + 16)
    rows = (k + per_row - 1) // per_row
    frame = np.zeros((rows * (side + 16) + 16, 1024), np.uint8)
    rng = np.random.default_rng(1)
    boxes = []
    for j in range(k):
        x, y = 16 + (j % per_row) * (side + 16), 16 + (j // per_row) * (side + 16)
        frame[y:y + side, x:x + side] = F.image_of(H[j], rng, (side, side))
        boxes.append(((x, y, side, side), j))
    return boxes, frame


def test_otsu_on_designed_units(insp):
    """Histograms of the adversarial Otsu families (exact ties, lone pixels, spikes) at 64 x 64 pixels on the general
    kernel with blur and morphology off, and flat patches with a step on the segmentation kernel: every unit equals
    the oracle."""
    rng = np.random.default_rng(17)
    H, _ = F.mixed(rng, 12)
    H = np.stack([rng.multinomial(4096, h / h.sum()) for h in H])
    boxes, frame = designed_units(H, 64)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    full_check(insp, frame[None], boxes, dict(gaussian_blur=0, morph_kernel=0))
    # flat patches with a step, default configuration
    rects = [b for b, _ in boxes[:48]]
    frames = np.stack([synth.make_frame(2400 + i, rects, H=frame.shape[0], W=1024, inset=4, max_discs=3)
                       for i in range(2)])
    for i, (x, y, w, h) in enumerate(rects):
        frames[0, y:y + h, x:x + w] = 40 + (i % 7) * 20
        frames[0, y + h // 2:y + h, x:x + w] += np.uint8(1 + i % 5)
    bx = [(r, i) for i, r in enumerate(rects)]
    insp.configure(Grid(boxes=bx), is_reference=True)
    prof = seg_profile(insp, 2)
    full_check(insp, frames, bx, {}, prof=prof)
    assert int(prof.count_nonzero()) > 0


# ---- 4. the general kernel --------------------------------------------------------------------------------------------

GENERAL = [dict(seg_method='adaptive', adapt_block=11, adapt_C=5), dict(gaussian_blur=0, morph_kernel=0),
           dict(gaussian_blur=5, morph_kernel=5)]


@pytest.mark.parametrize("ki", range(len(GENERAL)))
def test_general_kernel(insp, ki):
    kw = GENERAL[ki]
    boxes, _, bottom = shelf_layout(G1, 1008)
    n = frames_for(len(G1), sm_count())
    frames = make_frames(boxes, n, bottom + 8, 1024, 2500 + ki)
    insp.configure(Grid(boxes=boxes, exclusions=EXCL), is_reference=True)
    if kw.get('seg_method') == 'adaptive':
        # the adaptive mean is a float32 Gaussian (test_gpu_unit_sequences.py allows pixel differences against cv2):
        # here only the full call is the yardstick
        import torch
        p = vi_b200.default_params(**kw)
        ft = torch.from_numpy(frames).cuda()
        o = outs(insp, n)
        rec, seg = segment(insp, ft, p, **o)
        check_against_inspect(insp, ft, p, rec, seg, host(o))
        return
    full_check(insp, frames, boxes, kw, excl=EXCL, is_reference=True)


def test_general_kernel_on_frames_one_byte_off(insp):
    import torch
    boxes, _, bottom = shelf_layout(G1, 1008)
    n, H, W = 8, bottom + 8, 1024
    frames = make_frames(boxes, n, H, W, 2600)
    buf = torch.zeros(n * H * W + 1, dtype=torch.uint8, device="cuda")
    view = buf[1:].view(n, H, W)
    view.copy_(torch.from_numpy(frames).cuda())
    insp.configure(Grid(boxes=boxes), is_reference=True)
    full_check(insp, frames, boxes, {}, ft=view)


# ---- 5. the arena kernel ----------------------------------------------------------------------------------------------

def test_arena_kernel(insp):
    """ARENA_UNITS (G1 and 640 x 480) plus a 2048 x 1500 unit, many units per CTA."""
    units = ARENA_UNITS + [(2048, 1500, 3)]
    boxes, _, bottom = shelf_layout(units, 2100)
    n = frames_for(len(units), sm_count())
    frames = make_frames(boxes, n, bottom + 8, 2112, 2700)
    insp.configure(Grid(boxes=boxes, exclusions=EXCL), is_reference=True)
    full_check(insp, frames, boxes, {}, excl=EXCL, is_reference=True)


# ---- 6. outputs the call never writes ---------------------------------------------------------------------------------

def test_defect_outputs_stay_untouched(insp):
    """Defect bits and a blob table switched on for vi_inspect_batch keep their sentinel through segment_batch."""
    import torch
    boxes, _, bottom = shelf_layout(G1, 1008)
    frames = make_frames(boxes, 4, bottom + 8, 1024, 2800)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    n = frames.shape[0]
    dbits = torch.full((n * insp.packed_bytes,), SENT, dtype=torch.uint8, device="cuda")
    tab = torch.full((n * insp.n_units, 8, 40), SENT, dtype=torch.uint8, device="cuda")
    vi_b200._lib.check(insp._lib.vi_set_packed_mask_output(insp._ctx, None, C.c_void_p(dbits.data_ptr())))
    vi_b200._lib.check(insp._lib.vi_set_defect_blob_output(insp._ctx, C.c_void_p(tab.data_ptr()), 8))
    ft = torch.from_numpy(frames).cuda()
    rec = torch.empty((n * insp.n_units, 64), dtype=torch.uint8, device="cuda")
    seg = torch.empty(n * insp.unit_pixels, dtype=torch.uint8, device="cuda")
    vi_b200._lib.check(insp._lib.vi_segment_batch(insp._ctx, ft.data_ptr(), n, 1024, frames.shape[1], 1024,
                                                  1024 * frames.shape[1], C.byref(vi_b200.default_params()),
                                                  seg.data_ptr(), rec.data_ptr(), None))
    torch.cuda.synchronize()
    assert (dbits == SENT).all() and (tab == SENT).all()
    r = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    assert (r['status'] == vi_b200.STATUS_SEGMENTED).all()


# ---- 7. the host call -------------------------------------------------------------------------------------------------

def test_host_call_equals_the_device_call(insp, monkeypatch):
    import torch
    boxes, _, bottom = shelf_layout(G1, 1008)
    frames = make_frames(boxes, 12, bottom + 8, 1024, 2900)
    insp.configure(Grid(boxes=boxes, exclusions=EXCL), is_reference=True)
    p = vi_b200.default_params()
    o = outs(insp, 12)
    drec, dseg = segment(insp, torch.from_numpy(frames).cuda(), p, **o)
    bits = o['seg_bits'].cpu().numpy()
    monkeypatch.setenv("VI_HOST_CHUNK", "2")
    for fmt in ("bytes", "packed", "none"):
        hrec, hseg = insp.segment_batch_host(frames, p, mask_format=fmt)
        for f in vi_b200.RECORD_DTYPE.names:
            if f != 'n_runs':
                assert hrec.reshape(drec.shape)[f].tobytes() == drec[f].tobytes(), (fmt, f)
        if fmt == "bytes":
            assert np.array_equal(hseg, dseg.reshape(-1))
        elif fmt == "packed":
            assert np.array_equal(hseg, bits)
        else:
            assert hseg is None
    from vi_b200 import segmentation
    srec, smasks = segmentation.segment_batch(frames[:3], Grid(boxes=boxes, exclusions=EXCL), p, is_reference=True)
    assert srec.shape == (3, len(boxes)) and (srec['status'] == vi_b200.STATUS_SEGMENTED).all()
    for fi in range(3):
        segs = insp.split_masks(dseg[fi])
        assert all(np.array_equal(a, b) for a, b in zip(smasks[fi], segs))


# ---- 8. arguments -----------------------------------------------------------------------------------------------------

def test_argument_checks(insp):
    import torch
    lib, ctx = insp._lib, insp._ctx
    p = C.byref(vi_b200.default_params())
    rec = torch.empty((4, 64), dtype=torch.uint8, device="cuda")
    seg = torch.empty(1 << 16, dtype=torch.uint8, device="cuda")
    fr = torch.zeros((1, 64, 64), dtype=torch.uint8, device="cuda")
    assert lib.vi_segment_batch(ctx, fr.data_ptr(), 1, 64, 64, 64, 4096, p, seg.data_ptr(), rec.data_ptr(), None) == -1  # no grid
    insp.set_grid([(0, 0, 32, 32), (32, 32, 32, 32)])
    assert lib.vi_segment_batch(None, fr.data_ptr(), 1, 64, 64, 64, 4096, p, seg.data_ptr(), rec.data_ptr(), None) == -1
    assert lib.vi_segment_batch(ctx, None, 1, 64, 64, 64, 4096, p, seg.data_ptr(), rec.data_ptr(), None) == -1
    assert lib.vi_segment_batch(ctx, fr.data_ptr(), 1, 64, 64, 64, 4096, p, seg.data_ptr(), None, None) == -1
    assert lib.vi_segment_batch(ctx, fr.data_ptr(), 0, 64, 64, 64, 4096, p, seg.data_ptr(), rec.data_ptr(), None) == -1
    assert lib.vi_segment_batch(ctx, fr.data_ptr(), 1, 48, 64, 64, 4096, p, seg.data_ptr(), rec.data_ptr(), None) == -1
    assert lib.vi_segment_batch(ctx, fr.data_ptr(), 1, 64, 64, 32, 4096, p, seg.data_ptr(), rec.data_ptr(), None) == -1
    assert lib.vi_segment_batch(ctx, fr.data_ptr(), 1, 64, 64, 64, 4096, None, seg.data_ptr(), rec.data_ptr(), None) == -1
    bad = vi_b200.default_params(median_ksize=5)
    assert lib.vi_segment_batch(ctx, fr.data_ptr(), 1, 64, 64, 64, 4096, C.byref(bad), seg.data_ptr(), rec.data_ptr(), None) == -3
    hf = np.zeros((1, 64, 64), np.uint8)
    hrec = np.empty(2, vi_b200.RECORD_DTYPE)
    assert lib.vi_segment_batch_host(ctx, hf.ctypes.data, 1, 64, 64, 64, 4096, p, 3, None, hrec.ctypes.data) == -1
    assert lib.vi_segment_batch_host(ctx, hf.ctypes.data, 1, 64, 64, 64, 4096, p, 2, None, None) == -1
    with pytest.raises(TypeError):
        insp.segment_batch(torch.zeros((64, 64), dtype=torch.uint8, device="cuda"))
    with pytest.raises(ValueError):
        insp.segment_batch(fr, seg_masks=seg[:10])
    assert lib.vi_segment_batch(ctx, fr.data_ptr(), 1, 64, 64, 64, 4096, p, seg.data_ptr(), rec.data_ptr(), None) == 0
    torch.cuda.synchronize()


# ---- 9. the self-checked build ----------------------------------------------------------------------------------------

def test_checked_build_over_segment_batches():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    from vi_b200 import _build
    _build.build(checked=True)
    env = dict(os.environ, VI_B200_LIB="checked")
    res = subprocess.run([sys.executable, os.path.join(root, "tests", "checked_segment_run.py")], env=env,
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "check_word 0" in res.stdout, res.stdout + res.stderr
