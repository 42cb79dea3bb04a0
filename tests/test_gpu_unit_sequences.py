"""Sequences of units of different sizes on one CTA, and units at the size bound, against the cv2 oracle.

The inspection kernel is persistent: it launches min(units, CTAs) CTAs and CTA b runs units b, b + gridDim.x, ...
(vi_unit.cuh: vi_unit_kernel).  The shared-memory layout or global arena, the per-CTA L2 scratch (dirty-cell plane,
blur planes, run-table overflow, adaptive float plane), the mbarrier parity and, in the default-configuration kernel,
the asynchronous gather of the next unit's crop all carry over from one unit to the next.  The grids here are ragged
and their unit count does not divide the CTA count, so a CTA meets a small unit after a large one and the reverse;
every test asserts that coverage from the uid -> CTA map before it compares.

Run on the B200 box: python -m pytest tests/test_gpu_unit_sequences.py -m gpu"""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

from oracle import ref_cv2 as R
from oracle import restate as S
import vi_b200
from vi_b200 import synth
from vi_b200.grid import Grid

# BASELINE configs[3]'s exclusions: P7 runs at every unit size (clipped to the smaller units)
EXCL = [{'shape': 'rect', 'x': 50, 'y': 60, 'w': 70, 'h': 30}, {'shape': 'circle', 'cx': 200, 'cy': 180, 'r': 25}]

# G1 (w, h, byte phase x0 & 15).  Its largest unit (316 x 315) gives the default kernel's tensor-box gather tiles of
# 3 x 112 B by 160 rows in 2 row blocks; every unit but 3 x 3 (narrower than 4) takes the boxes.
G1 = [(3, 3, 5), (13, 21, 1), (36, 40, 15), (40, 33, 7), (96, 96, 3), (150, 141, 9), (200, 150, 0),
      (316, 315, 11), (300, 200, 13), (97, 111, 2), (64, 64, 4), (250, 60, 6), (20, 300, 14)]
# G2: no tile split of its largest width / height (500 x 330) fits the 71,200 B staging area, so the default kernel
# gathers by row copies: 150x230, 100x330, 96x96, 316x200, 36x40, 200x150 and 380x80 take them; 3x3, 2x330, 13x21
# (gray pitch beyond the staging pitch) and 500x60 (wider than 384) load synchronously.  (A taller largest unit, such
# as 2 x 400, leaves the median stage's lattice no room in shared memory: the general kernel would run instead.)
G2 = [(3, 3, 0), (13, 21, 5), (150, 230, 9), (500, 60, 3), (100, 330, 12), (96, 96, 7),
      (316, 200, 1), (36, 40, 14), (200, 150, 6), (2, 330, 11), (380, 80, 2)]


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def frames_for(n_units, sms):
    """Enough images that every CTA (one per SM) runs at least 4 units."""
    return math.ceil(4 * sms / n_units)


def assert_sequences(shapes, n_images, ctas):
    """The uid -> CTA map of the persistent kernel (CTA b runs uids b, b + ctas, ...): every CTA runs at least 3
    units, and some CTA goes from a larger unit to a smaller one and some from a smaller one to a larger one."""
    n_units = len(shapes)
    total = n_images * n_units
    nb = min(total, ctas)
    area = [w * h for w, h in shapes]
    down = up = 0
    for b in range(nb):
        seq = [area[u % n_units] for u in range(b, total, nb)]
        assert len(seq) >= 3, (b, len(seq))
        down += sum(p > q for p, q in zip(seq, seq[1:]))
        up += sum(p < q for p, q in zip(seq, seq[1:]))
    assert down > 0 and up > 0, (down, up)


def shelf_layout(units, wlim, gap=6):
    """Boxes for (w, h, phase) units, left to right on shelves no wider than wlim, each at x0 & 15 == phase.
    Returns (boxes as ((x, y, w, h), idx), right edge, bottom edge)."""
    boxes, x, y, shelf, right = [], 0, gap, 0, 0
    for i, (w, h, ph) in enumerate(units):
        x0 = (x + gap + 15) // 16 * 16 + ph
        if x0 + w + gap > wlim:
            y += shelf + gap
            shelf = 0
            x0 = 16 + ph
        boxes.append(((x0, y, w, h), i))
        x = x0 + w
        shelf = max(shelf, h)
        right = max(right, x0 + w)
    return boxes, right, y + shelf


def make_frames(boxes, n, H, W, seed0, **kw):
    rects = [b for b, _ in boxes]
    return np.stack([synth.make_frame(seed0 + i, rects, H=H, W=W, inset=kw.get('inset', 5), jitter=2,
                                      max_discs=kw.get('max_discs', 4)) for i in range(n)])


def ref_centroids(frame, boxes, rp):
    recs, _, _ = R.inspect_frame(frame, boxes, rp, EXCL, None, True)
    return {i: (r['cx'], r['cy']) for i, r in enumerate(recs) if r['cx'] == r['cx']}


def run_device(insp, frames_t, params, **outs):
    import torch
    rec, seg, dfm = insp.inspect_batch(frames_t, params, **outs)
    torch.cuda.synchronize()
    n = frames_t.shape[0]
    rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(n, insp.n_units)
    return rec, seg.cpu().numpy().reshape(n, -1), dfm.cpu().numpy().reshape(n, -1)


def assert_records_equal(a, b, skip=()):
    """Field by field, bit for bit (NaN centroids of units without a seg component included)."""
    for f in vi_b200.RECORD_DTYPE.names:
        if f not in skip:
            assert a[f].tobytes() == b[f].tobytes(), f


def blur_k(kw):
    b = kw.get('gaussian_blur', 3)
    k = b if b % 2 == 1 else b + 1
    return k if b > 0 and k > 1 else 0


def check_oracle(insp, frames, boxes, kw, refc, rec, seg, dfm, tol=0.0):
    """Every unit of every image against R.inspect_frame: both masks bit for bit, the record fields, cx / cy
    bit-equal, otsu_t against Otsu of the blurred crop.  tol > 0 (adaptive mean, a float32 Gaussian): up to tol of
    the seg-mask pixels may differ; units whose seg mask differs skip the other comparisons.  Returns the records
    of the oracle."""
    rp = R.Params(**kw)
    k = blur_k(kw)
    bad = tot = 0
    out = []
    for fi in range(len(frames)):
        recs, osegs, odefs = R.inspect_frame(frames[fi], boxes, rp, EXCL, refc, False)
        out.append(recs)
        segs = insp.split_masks(seg[fi]); defs = insp.split_masks(dfm[fi])
        for u, o in enumerate(recs):
            r = rec[fi, u]
            assert r['image'] == fi and r['unit'] == u
            nbad = int((segs[u] != osegs[u]).sum())
            bad += nbad; tot += osegs[u].size
            if nbad:
                assert tol > 0, (kw, fi, u, 'seg', nbad)
                continue
            want = odefs[u] if odefs[u] is not None else np.zeros_like(defs[u])
            assert np.array_equal(defs[u], want), (kw, fi, u, 'defect', int((defs[u] != want).sum()))
            for f in ('seg_area', 'roi_area', 'defect_area', 'n_kept', 'status', 'dx', 'dy'):
                assert r[f] == o[f], (kw, fi, u, f, r[f], o[f])
            assert np.array_equal(np.float64([r['cx'], r['cy']]).view(np.int64),
                                  np.float64([o['cx'], o['cy']]).view(np.int64)), (kw, fi, u, 'centroid')
            if kw.get('seg_method', 'otsu') != 'adaptive':
                (x, y, w, h), _ = boxes[u]
                crop = np.ascontiguousarray(frames[fi, y:y + h, x:x + w])
                assert r['otsu_t'] == R.otsu_threshold(cv2.GaussianBlur(crop, (k, k), 0) if k else crop), (kw, fi, u, 'otsu_t')
    assert bad <= tol * tot, (kw, bad, tot)
    return out


def configure(insp, frames, boxes, kw):
    """Exclusions and the centroid shift against frame 0 (the reference frame's centroids)."""
    refc = ref_centroids(frames[0], boxes, R.Params(**kw))
    insp.configure(Grid(boxes=boxes, exclusions=EXCL, ref_centroids=refc), is_reference=False)
    return refc


@pytest.fixture(autouse=True)
def opencv_otsu_scan():
    """The oracle's Otsu threshold from OpenCV's C++ scan, which the kernels follow.  The 3 x 3 units' blurred
    histograms are often mirror-symmetric (an exact tie), and the IPP routine the cv2 wheel dispatches to by default
    breaks such ties differently (test_gpu_parity.py: test_otsu_threshold_near_ties)."""
    ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    yield
    cv2.ipp.setUseIPP(ipp)


@pytest.fixture
def insp():
    i = vi_b200.Inspector(0)
    yield i
    i.close()


def g1_frames(n, seed0=100):
    boxes, right, bottom = shelf_layout(G1, 1008)
    return boxes, make_frames(boxes, n, bottom + 8, 1024, seed0)


# ---- 1. the default-configuration kernel (SPEC), tensor-box gather --------------------------------------------------

def test_spec_box_gather_over_ragged_sequences(insp):
    """G1 on 16-byte aligned frames, default parameters: tensor boxes for every unit but 3 x 3, which loads
    synchronously in the middle of the sequences."""
    import torch
    sms = sm_count()
    n = frames_for(len(G1), sms)
    boxes, frames = g1_frames(n)
    assert_sequences([(w, h) for w, h, _ in G1], n, sms)
    assert all(b[0][0] & 15 == ph for b, (_, _, ph) in zip(boxes, G1))
    refc = configure(insp, frames, boxes, {})
    rec, seg, dfm = run_device(insp, torch.from_numpy(frames).cuda(), vi_b200.default_params())
    check_oracle(insp, frames, boxes, {}, refc, rec, seg, dfm)
    assert (rec['dx'] != 0).any() or (rec['dy'] != 0).any()


def test_spec_box_gather_on_a_strided_view(insp):
    """G1 on a view [:, :H, :W] of [n, H + 32, Wp] frames: aligned row pitch, image stride beyond pitch x H, and
    W = 9 (mod 16), with a unit flush against the right and bottom edges -- the boxes run past the frame edge and
    are zero-filled."""
    import torch
    sms = sm_count()
    n = frames_for(len(G1), sms)
    boxes, right, bottom = shelf_layout(G1, 1008)
    W = (right + 300 + 15) // 16 * 16 + 9
    H = bottom + 8
    (_, _, w9, h9), i9 = boxes[8]
    assert (w9, h9) == (300, 200)
    boxes[8] = ((W - 300, H - 200, 300, 200), i9)                     # x0 & 15 == 13, x + w == W, y + h == H
    assert W % 16 == 9 and boxes[8][0][0] & 15 == 13
    assert_sequences([(w, h) for w, h, _ in G1], n, sms)
    frames = make_frames(boxes, n, H, W, 300)
    Wp = (W + 15) // 16 * 16 + 16
    full = torch.zeros((n, H + 32, Wp), dtype=torch.uint8, device="cuda")
    view = full[:, :H, :W]
    view.copy_(torch.from_numpy(frames).cuda())
    assert view.stride(1) % 16 == 0 and view.stride(0) > view.stride(1) * H and view.data_ptr() % 16 == 0
    refc = configure(insp, frames, boxes, {})
    rec, seg, dfm = run_device(insp, view, vi_b200.default_params())
    check_oracle(insp, frames, boxes, {}, refc, rec, seg, dfm)


def test_spec_empty_rois_interleave_sync_and_async_arrivals(insp):
    """erode_px=40: the small units' ROIs are empty and return before the next unit's gather is issued (that unit
    loads synchronously), the large ones issue it."""
    import torch
    sms = sm_count()
    n = frames_for(len(G1), sms)
    boxes, frames = g1_frames(n, seed0=500)
    assert_sequences([(w, h) for w, h, _ in G1], n, sms)
    kw = dict(erode_px=40)
    refc = configure(insp, frames, boxes, kw)
    rec, seg, dfm = run_device(insp, torch.from_numpy(frames).cuda(), vi_b200.default_params(**kw))
    check_oracle(insp, frames, boxes, kw, refc, rec, seg, dfm)
    st = rec['status']
    assert (st == vi_b200.STATUS_ROI_EMPTY).any() and (st != vi_b200.STATUS_ROI_EMPTY).any()


# ---- 2. SPEC, row-copy gather ------------------------------------------------------------------------------------------

def test_spec_row_gather_over_ragged_sequences(insp):
    import torch
    sms = sm_count()
    n = frames_for(len(G2), sms)
    boxes, right, bottom = shelf_layout(G2, 1008)
    assert all(b[0][0] & 15 == ph for b, (_, _, ph) in zip(boxes, G2))
    frames = make_frames(boxes, n, bottom + 8, 1024, 700)
    assert_sequences([(w, h) for w, h, _ in G2], n, sms)
    refc = configure(insp, frames, boxes, {})
    rec, seg, dfm = run_device(insp, torch.from_numpy(frames).cuda(), vi_b200.default_params())
    check_oracle(insp, frames, boxes, {}, refc, rec, seg, dfm)


# ---- 3. the general kernel over G1 -------------------------------------------------------------------------------------

GENERAL = [dict(gaussian_blur=5, morph_kernel=5), dict(gaussian_blur=0, morph_kernel=0),
           dict(seg_method='adaptive', adapt_block=11, adapt_C=5), dict(defect_method='canny', threshold=24)]


@pytest.mark.parametrize("ki", range(len(GENERAL)))
def test_general_kernel_over_ragged_sequences(insp, ki):
    """Non-default blur / morphology, adaptive (<= 1e-4 of the seg pixels, the bound test_segment_cell_adaptive
    states) and Canny: the general instantiation, many units per CTA."""
    import torch
    kw = GENERAL[ki]
    sms = sm_count()
    n = frames_for(len(G1), sms)
    boxes, frames = g1_frames(n, seed0=900 + 100 * ki)
    assert_sequences([(w, h) for w, h, _ in G1], n, sms)
    refc = configure(insp, frames, boxes, kw)
    rec, seg, dfm = run_device(insp, torch.from_numpy(frames).cuda(), vi_b200.default_params(**kw))
    check_oracle(insp, frames, boxes, kw, refc, rec, seg, dfm, tol=1e-4 if 'adapt_block' in kw else 0.0)


def test_general_kernel_optional_outputs_equal_the_default_kernel(insp):
    """Labels, seg stats and packed mask bits turn the default configuration over to the general kernel: its masks
    and records equal the default kernel's on the same frames, and every image's labels, stats and packed bits
    match what they restate."""
    import torch
    sms = sm_count()
    n = frames_for(len(G1), sms)
    boxes, frames = g1_frames(n, seed0=1400)
    assert_sequences([(w, h) for w, h, _ in G1], n, sms)
    refc = configure(insp, frames, boxes, {})
    d = torch.from_numpy(frames).cuda()
    p = vi_b200.default_params()
    rec0, seg0, dfm0 = run_device(insp, d, p)
    check_oracle(insp, frames, boxes, {}, refc, rec0, seg0, dfm0)
    nu = insp.n_units
    lab = torch.full((n * insp.unit_pixels,), -1, dtype=torch.int32, device="cuda")
    stats = torch.full((n * nu, 3), -1, dtype=torch.int64, device="cuda")
    sb = torch.zeros(n * insp.packed_bytes, dtype=torch.uint8, device="cuda")
    db = torch.zeros(n * insp.packed_bytes, dtype=torch.uint8, device="cuda")
    rec, seg, dfm = run_device(insp, d, p, labels=lab, seg_stats=stats, seg_bits=sb, defect_bits=db)
    assert np.array_equal(seg, seg0) and np.array_equal(dfm, dfm0)
    assert_records_equal(rec, rec0, skip=('n_ambiguous', 'n_runs'))     # diagnostics: counted by whichever passes ran
    lab = lab.cpu().numpy().reshape(n, -1)
    stats = stats.cpu().numpy().reshape(n, nu, 3)
    sb, db = sb.cpu().numpy(), db.cpu().numpy()
    for fi in range(n):
        segs = insp.split_masks(seg[fi]); defs = insp.split_masks(dfm[fi]); labs = insp.split_masks(lab[fi])
        for u in range(nu):
            er = cv2.erode(((segs[u] > 0) * 255).astype(np.uint8), None, iterations=6)
            lab_ref, _ = S.label8(er)
            assert np.array_equal(labs[u], lab_ref), (fi, u, 'labels')
            ys, xs = np.nonzero(segs[u])
            assert tuple(stats[fi, u]) == (len(xs), int(xs.sum()), int(ys.sum())), (fi, u, 'seg_stats')
        for a, b in zip(insp.unpack_masks(sb, fi), segs):
            assert np.array_equal(a, b), (fi, 'seg bits')
        for a, b in zip(insp.unpack_masks(db, fi), defs):
            assert np.array_equal(a, b), (fi, 'defect bits')


def test_general_kernel_on_frames_one_byte_off(insp):
    """Default parameters on frames whose base pointer is one byte past an aligned address: the general kernel's
    scalar crop load."""
    import torch
    sms = sm_count()
    n = frames_for(len(G1), sms)
    boxes, frames = g1_frames(n, seed0=1600)
    assert_sequences([(w, h) for w, h, _ in G1], n, sms)
    refc = configure(insp, frames, boxes, {})
    buf = torch.zeros(frames.size + 16, dtype=torch.uint8, device="cuda")
    d = buf[1:1 + frames.size].view(frames.shape)
    d.copy_(torch.from_numpy(frames).cuda())
    assert d.data_ptr() % 16 == 1
    rec, seg, dfm = run_device(insp, d, vi_b200.default_params())
    check_oracle(insp, frames, boxes, {}, refc, rec, seg, dfm)


# ---- 4. the arena kernel (GMEM) over many units -------------------------------------------------------------------------

ARENA = [dict(), dict(defect_method='canny', threshold=24), dict(seg_method='adaptive', adapt_block=11, adapt_C=5),
         dict(gaussian_blur=7, morph_kernel=5)]
ARENA_UNITS = G1 + [(640, 480, 8)]


@pytest.mark.parametrize("ki", range(len(ARENA)))
def test_arena_kernel_over_ragged_sequences(insp, ki):
    """G1 plus one 640 x 480 unit, which does not fit one SM's shared memory: the whole grid runs over the per-CTA
    global arena, which every CTA reuses for at least 3 units."""
    import torch
    kw = ARENA[ki]
    sms = sm_count()
    n = frames_for(len(ARENA_UNITS), sms)
    boxes, right, bottom = shelf_layout(ARENA_UNITS, 1008)
    frames = make_frames(boxes, n, bottom + 8, 1024, 2000 + 100 * ki, inset=12)
    assert_sequences([(w, h) for w, h, _ in ARENA_UNITS], n, sms)
    refc = configure(insp, frames, boxes, kw)
    rec, seg, dfm = run_device(insp, torch.from_numpy(frames).cuda(), vi_b200.default_params(**kw))
    check_oracle(insp, frames, boxes, kw, refc, rec, seg, dfm, tol=1e-4 if 'adapt_block' in kw else 0.0)


def test_arena_compat_calls(insp):
    """The per-unit calls on a 640 x 480 crop (arena path) with the configurations the batch tests above leave to
    them: segment_cell adaptive, blur 5 / morph 5, blur 0; detect_defects with Canny."""
    box = (10, 12, 640, 480)
    fr = synth.make_frame(77, [box], H=500, W=672, inset=30, max_discs=6)
    crop = fr[12:492, 10:650].copy()
    got = insp.segment_cell(crop, vi_b200.default_params(seg_method='adaptive', adapt_block=11, adapt_C=5))
    want = R.segment_cell(crop, method='adaptive', adapt_block=11, adapt_C=5)
    assert int((got != want).sum()) <= 1e-4 * want.size
    for kw in (dict(gaussian_blur=5, morph_kernel=5), dict(gaussian_blur=0, morph_kernel=0)):
        got, t = insp.segment_cell(crop, vi_b200.default_params(**kw), return_threshold=True)
        assert np.array_equal(got, R.segment_cell(crop, **kw)), kw
        k = blur_k(kw)
        assert t == R.otsu_threshold(cv2.GaussianBlur(crop, (k, k), 0) if k else crop), kw
    seg = R.segment_cell(crop)
    found = 0
    for thr, mn, r in ((24, 20, 6), (8, 0, 2)):
        info = {}
        ref = R.detect_defects(crop, seg, 'canny', thr, mn, r, info)
        got, rec = insp.detect_defects(crop, seg, vi_b200.default_params(defect_method='canny', threshold=thr, min_area=mn,
                                                                         erode_px=r), return_record=True)
        assert (ref is None) == (got is None), thr
        assert rec['n_kept'] == info['n_kept'] and rec['roi_area'] == int((info['roi'] > 0).sum())
        if ref is not None:
            found += 1
            assert np.array_equal(got, ref), (thr, int((got != ref).sum()))
            assert rec['defect_area'] == int((ref > 0).sum())
    assert found > 0


# ---- 5. the host-buffer call over G1 -------------------------------------------------------------------------------------

def covered_rows(boxes):
    iv = sorted((y, y + h) for (x, y, w, h), _ in boxes)
    rows = []
    for a, b in iv:
        if rows and a <= rows[-1][1]:
            rows[-1][1] = max(rows[-1][1], b)
        else:
            rows.append([a, b])
    return sum(b - a for a, b in rows)


def test_host_buffer_call_over_ragged_sequences(insp, monkeypatch):
    """G1 through the host-buffer call in chunks large enough that every CTA of a chunk's launch runs at least 3
    units, and at least two chunks per slot (3 slots), byte and packed masks: equal to the device call; the upload
    size is the merged covered rows x W x n."""
    import torch
    sms = sm_count()
    chunk = math.ceil(3 * sms / len(G1))
    n = 6 * chunk
    boxes, frames = g1_frames(n, seed0=1800)
    assert_sequences([(w, h) for w, h, _ in G1], chunk, sms)
    refc = configure(insp, frames, boxes, {})
    W = frames.shape[2]
    assert insp._lib.vi_host_upload_bytes(insp._ctx, n, W) == covered_rows(boxes) * W * n
    p = vi_b200.default_params()
    rec_d, seg_d, dfm_d = run_device(insp, torch.from_numpy(frames).cuda(), p)
    check_oracle(insp, frames, boxes, {}, refc, rec_d, seg_d, dfm_d)
    monkeypatch.setenv("VI_HOST_CHUNK", str(chunk))
    rec_h, seg_h, dfm_h = insp.inspect_batch_host(frames, p)
    assert np.array_equal(seg_h.reshape(n, -1), seg_d) and np.array_equal(dfm_h.reshape(n, -1), dfm_d)
    assert_records_equal(rec_h, rec_d.reshape(-1))
    rec_p, seg_p, dfm_p = insp.inspect_batch_host(frames, p, mask_format="packed")
    assert_records_equal(rec_p, rec_h)
    for fi in range(n):
        for a, b in zip(insp.unpack_masks(seg_p, fi), insp.split_masks(seg_d[fi])):
            assert np.array_equal(a, b), fi
        for a, b in zip(insp.unpack_masks(dfm_p, fi), insp.split_masks(dfm_d[fi])):
            assert np.array_equal(a, b), fi


# ---- 6. units at the size bound -------------------------------------------------------------------------------------------

def device_mem_used():
    import torch
    free, total = torch.cuda.mem_get_info(0)
    return total - free


def big_and_small_frame(seed, big, small, H, W, inset):
    """A frame with the plate of the big units at `inset` and the small units' own plates pasted over it."""
    fr = synth.make_frame(seed, big, H=H, W=W, inset=inset, max_discs=3)
    other = synth.make_frame(seed + 1000, small, H=H, W=W, inset=5, max_discs=2)
    for (x, y, w, h) in small:
        fr[y:y + h, x:x + w] = other[y:y + h, x:x + w]
    return fr


def run_bound(boxes, frames, kw=None):
    """One Inspector for the call (its per-CTA scratch is about 25 GB at the bound), closed afterwards.  Prints the
    device memory in use while it exists."""
    import torch
    kw = kw or {}
    before = device_mem_used()
    insp = vi_b200.Inspector(0)
    try:
        refc = configure(insp, frames, boxes, kw)
        d = torch.from_numpy(frames).cuda()
        rec, seg, dfm = run_device(insp, d, vi_b200.default_params(**kw))
        print(f"\n[bound] units {[b[2:] for b, _ in boxes][:3]}... x {len(boxes)}: device memory in use "
              f"{(device_mem_used() - before) / 2**30:.2f} GiB")
        del d
        return check_oracle(insp, frames, boxes, kw, refc, rec, seg, dfm), rec
    finally:
        insp.close()
        torch.cuda.empty_cache()


def test_unit_of_2_24_pixels_near_the_moment_bound():
    """A 4096 x 4096 unit (2^24 px) on a bright field of 255 around a dark plate: the histogram moment sum i * h_i,
    summed in 32 bits, is close to 2^32."""
    box = (0, 8, 4096, 4096)
    frames = np.stack([synth.make_frame(s, [box], H=4112, W=4096, inset=1400, max_discs=3) for s in (60, 61)])
    frames[frames > 160] = 255
    moment = int(cv2.GaussianBlur(frames[0, 8:4104], (3, 3), 0).astype(np.int64).sum())
    assert 0.9 * 2**32 < moment < 2**32
    recs, rec = run_bound([(box, 0)], frames)
    assert rec['roi_area'].min() > 0


@pytest.mark.parametrize("wh", [(2048, 8192), (4096, 3000), (4096, 1), (1, 8192)])
def test_units_at_the_size_bound(wh):
    """The tallest unit (2048 x 8192), a whole 4096 x 3000 frame (with the grid.json plates in it), and the
    thinnest ones (4096 x 1, 1 x 8192), each over 2 frames against the oracle."""
    w, h = wh
    if wh == (4096, 3000):
        plates = [b for b, _ in vi_b200.generate_grid((251, 232, 316, 315), 4, 6, 2, 1, 133, 136, 252, 0)]
        frames = np.stack([synth.make_frame(s, plates) for s in (62, 63)])
        box = (0, 0, 4096, 3000)
    else:
        box = (16 if w < 4096 else 0, 8, w, h)
        frames = np.stack([synth.make_frame(s, [box], H=h + 16, W=max(w + 32, 64), inset=min(64, max(0, min(w, h) // 4)),
                                            max_discs=3) for s in (64, 65)])
    run_bound([(box, 0)], frames)


def test_a_2_24_pixel_unit_among_small_units():
    """One 4096 x 4096 unit among 60 small overlapping ones, 2 images: the scratch budget cuts the grid to fewer CTAs
    than SMs (36 on a 148-SM B200), each of which strides through about 3 units, small ones before and after the
    big one on the CTAs that run it."""
    rng = np.random.default_rng(8)
    small = []
    for i in range(60):
        w, h, _ = G1[i % len(G1)]
        small.append((int(rng.integers(0, 4096 - w)), int(rng.integers(0, 4112 - h)), w, h))
    big = (0, 8, 4096, 4096)
    boxes = [(r, i) for i, r in enumerate(small[:20] + [big] + small[20:])]
    frames = np.stack([big_and_small_frame(s, [big], small, 4112, 4096, 1200) for s in (66, 67)])
    run_bound(boxes, frames)


# ---- 7. the pixel bound holds per unit ------------------------------------------------------------------------------------

def test_ragged_grid_beyond_2_24_pixels_of_wmax_x_hmax():
    """A 4096 x 200 strip and a 200 x 8000 column are each within the bound; the grid's largest width times largest
    height (4096 x 8000) is not, and must not be what the bound is checked on."""
    strip, column = (0, 0, 4096, 200), (1000, 200, 200, 8000)
    rng = np.random.default_rng(9)
    small = []
    for i in range(13):
        w, h, _ = G1[i]
        small.append((int(rng.integers(0, 4096 - w)), int(rng.integers(0, 8200 - h)), w, h))
    boxes = [(r, i) for i, r in enumerate([strip] + small[:7] + [column] + small[7:])]
    frames = np.stack([big_and_small_frame(s, [strip, column], small, 8200, 4096, 20) for s in (68, 69)])
    recs, rec = run_bound(boxes, frames)
    assert rec['roi_area'][:, 0].min() > 0 and rec['roi_area'][:, 8].min() > 0
