"""The kept-defect-component table (vi_set_defect_blob_output, inspect_batch(defect_blobs=...),
inspect_batch_host(max_blobs=K)) against the cv2 oracle of tests/blob_oracle.py, on every kernel instantiation.

Every (image, unit) is compared field for field (cx / cy bit for bit) for its first min(n_kept, K) components.  The
device table is pre-filled with a sentinel, and every slot past min(n_kept, K) must still hold it: nothing is written
there, and nothing carries over from a CTA's earlier unit.

Run on the B200 box: python -m pytest tests/test_gpu_defect_blobs.py -m gpu"""
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
from vi_b200.grid import Grid
from test_gpu_unit_sequences import (ARENA_UNITS, EXCL, G1, assert_records_equal, assert_sequences, configure,
                                     frames_for, make_frames, shelf_layout, sm_count)

import blob_oracle as BO

SENT = 0xA5
# n_runs is a diagnostic: the largest run count of whichever labelling passes ran, and whether the hole fill's flood
# settles within its rounds (its reads of neighbour rows race) decides whether a background labelling runs at all
DIAG = ('n_runs',)
CONFIG5 = dict(threshold=8, min_area=0, erode_px=1)


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


def run(insp, frames, params, K=None, **outs):
    """One device batch; K: a sentinel-filled blob table [n*units, K, 40] is passed.  Returns host copies
    (records [n, units], seg, defect, raw blob table or None)."""
    import torch
    n = frames.shape[0]
    tab = None
    if K:
        tab = torch.full((n * insp.n_units, K, 40), SENT, dtype=torch.uint8, device="cuda")
    ft = frames if isinstance(frames, torch.Tensor) else torch.from_numpy(frames).cuda()
    rec, seg, dfm = insp.inspect_batch(ft, params, defect_blobs=tab, **outs)
    torch.cuda.synchronize()
    rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(n, insp.n_units)
    return rec, seg.cpu().numpy(), dfm.cpu().numpy(), (tab.cpu().numpy() if K else None)


def check_blobs(insp, frames, boxes, kw, rec, raw, K, excl=(), refc=None, sentinel=True):
    """Every unit's table against the oracle; returns the oracle's n_kept per (image, unit)."""
    rp = R.Params(**kw)
    nk = np.zeros(rec.shape, np.int64)
    for fi in range(len(frames)):
        _, osegs, _ = R.inspect_frame(frames[fi], boxes, rp, excl, refc, False)
        for u, ((x, y, w, h), _) in enumerate(boxes):
            crop = np.ascontiguousarray(frames[fi, y:y + h, x:x + w])
            want = BO.kept_defect_blobs(crop, osegs[u], **BO.params_kw(rp))
            assert rec[fi, u]['n_kept'] == len(want), (kw, fi, u, rec[fi, u]['n_kept'], len(want))
            got = insp.kept_blobs(rec, raw, fi, u)
            BO.assert_blobs_equal(got, want[:K], (kw, fi, u))
            if sentinel:
                uid = fi * insp.n_units + u
                assert (raw[uid, len(got):] == SENT).all(), (kw, fi, u, 'written past min(n_kept, K)')
            nk[fi, u] = len(want)
    return nk


def grid_json_frames(n, seed0=40):
    boxes = vi_b200.generate_grid((251, 232, 316, 315), 4, 6, 2, 1, 133, 136, 252, 0)
    return boxes, np.stack([synth.make_frame(seed0 + i, [b for b, _ in boxes], max_discs=6) for i in range(n)])


def salted(boxes, n, H, W, seed0, salt_of):
    """Frames of the given boxes; image i has salt noise of probability salt_of(i) in its plates."""
    rects = [b for b, _ in boxes]
    return np.stack([synth.make_frame(seed0 + i, rects, H=H, W=W, inset=5, jitter=2, max_discs=4, salt_p=salt_of(i))
                     for i in range(n)])


def dense_small(n_x=6, n_y=4):
    return [((32 + 128 * i, 32 + 128 * j, 96, 96), j * n_x + i) for j in range(n_y) for i in range(n_x)]


# ---- 1. the default-configuration kernel ------------------------------------------------------------------------------

def test_default_kernel_blobs_and_phase_profile(insp):
    """grid.json frames with discs, K = 64: every unit equal to the oracle.  The phase-profile buffer is written in the
    same configuration, which only the default-configuration (SPEC) kernel does: the blob table keeps it there."""
    import torch
    boxes, frames = grid_json_frames(3)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    prof = torch.zeros((3 * insp.n_units, 48), dtype=torch.int64, device="cuda")
    vi_b200._lib.check(insp._lib.vi_debug_set_profile(insp._ctx, C.c_void_p(prof.data_ptr())))
    try:
        rec, _, _, raw = run(insp, frames, vi_b200.default_params(), K=64)
    finally:
        vi_b200._lib.check(insp._lib.vi_debug_set_profile(insp._ctx, None))
    assert int(prof.count_nonzero()) > 0
    nk = check_blobs(insp, frames, boxes, {}, rec, raw, 64)
    assert nk.sum() > 20 and (nk == 0).any()


# ---- 2. nothing else changes ------------------------------------------------------------------------------------------

def test_blob_table_changes_no_other_output(insp, monkeypatch):
    """Records, byte masks, packed masks, labels and seg stats are identical with the table off and on: the default
    kernel, the general kernel with every optional output, and the host call in bytes and packed formats."""
    import torch
    boxes, _, bottom = shelf_layout(G1, 1008)
    frames = salted(boxes, 8, bottom + 8, 1024, 500, lambda i: 0.05 if i % 2 == 0 else 0.0)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    n = frames.shape[0]
    for kw in (dict(), CONFIG5):
        p = vi_b200.default_params(**kw)
        a = run(insp, frames, p)
        b = run(insp, frames, p, K=16)
        assert_records_equal(a[0], b[0], skip=DIAG)
        assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
        assert b[0]['n_kept'].sum() > 0

    def outs():
        return dict(labels=torch.empty(n * insp.unit_pixels, dtype=torch.int32, device="cuda"),
                    seg_stats=torch.empty((n * insp.n_units, 3), dtype=torch.int64, device="cuda"),
                    seg_bits=torch.empty(n * insp.packed_bytes, dtype=torch.uint8, device="cuda"),
                    defect_bits=torch.empty(n * insp.packed_bytes, dtype=torch.uint8, device="cuda"))
    p = vi_b200.default_params(**CONFIG5)
    oa, ob = outs(), outs()
    a = run(insp, frames, p, **oa)
    b = run(insp, frames, p, K=16, **ob)
    assert_records_equal(a[0], b[0], skip=DIAG)
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    for k in oa:
        assert torch.equal(oa[k], ob[k]), k
    monkeypatch.setenv("VI_HOST_CHUNK", "1")
    for fmt in ("bytes", "packed"):
        ha = insp.inspect_batch_host(frames, p, mask_format=fmt)
        hb = insp.inspect_batch_host(frames, p, mask_format=fmt, max_blobs=16)
        assert len(ha) == 3 and len(hb) == 4
        assert_records_equal(ha[0], hb[0], skip=DIAG)
        assert np.array_equal(ha[1], hb[1]) and np.array_equal(ha[2], hb[2])


# ---- 3. truncation and many components --------------------------------------------------------------------------------

@pytest.mark.parametrize("K", [1, 8, 1024])
def test_truncation_and_many_components(insp, K):
    """BASELINE configs[4] in miniature: 96 x 96 units, salt noise, threshold 8, min_area 0, erode 1.  n_kept exceeds
    K = 1 and 8; with K = 1024 some unit keeps more components than two masks of accumulators hold (57), so its table
    lives in the CTA's global scratch."""
    boxes = dense_small()
    frames = salted(boxes, 6, 576, 832, 700, lambda i: (0.02, 0.15, 0.3)[i % 3])
    insp.configure(Grid(boxes=boxes), is_reference=True)
    rec, _, _, raw = run(insp, frames, vi_b200.default_params(**CONFIG5), K=K)
    nk = check_blobs(insp, frames, boxes, CONFIG5, rec, raw, K)
    assert (nk > max(K, 8)).any() if K < 1024 else (nk > 2 * 1152 // 40).any()


# ---- 4. the general kernel --------------------------------------------------------------------------------------------

GENERAL = [dict(defect_method='canny'), dict(gaussian_blur=5, morph_kernel=5)]


@pytest.mark.parametrize("ki", range(len(GENERAL)))
def test_general_kernel_blobs(insp, ki):
    """Canny and blur / morph 5 on G1, with exclusions and the centroid shift; the second case also asks for labels,
    seg stats and packed bits next to the table."""
    import torch
    kw = GENERAL[ki]
    boxes, _, bottom = shelf_layout(G1, 1008)
    frames = make_frames(boxes, 10, bottom + 8, 1024, 900, max_discs=6)
    refc = configure(insp, frames, boxes, kw)
    n = frames.shape[0]
    outs = {}
    if ki == 1:
        outs = dict(labels=torch.empty(n * insp.unit_pixels, dtype=torch.int32, device="cuda"),
                    seg_stats=torch.empty((n * insp.n_units, 3), dtype=torch.int64, device="cuda"),
                    seg_bits=torch.empty(n * insp.packed_bytes, dtype=torch.uint8, device="cuda"),
                    defect_bits=torch.empty(n * insp.packed_bytes, dtype=torch.uint8, device="cuda"))
    rec, _, _, raw = run(insp, frames, vi_b200.default_params(**kw), K=32, **outs)
    assert (rec['dx'] != 0).any() or (rec['dy'] != 0).any()
    nk = check_blobs(insp, frames, boxes, kw, rec, raw, 32, excl=EXCL, refc=refc)
    assert nk.sum() > 0


# ---- 5. the arena kernel ----------------------------------------------------------------------------------------------

def test_arena_kernel_blobs_over_ragged_sequences(insp):
    """ARENA_UNITS plus a 2048 x 1500 unit, many units per CTA.  Image 0's large unit is salted so that it keeps more
    than 1024 components: its table truncates at K = 1024."""
    units = ARENA_UNITS + [(2048, 1500, 3)]
    boxes, _, bottom = shelf_layout(units, 2100)
    sms = sm_count()
    n = frames_for(len(units), sms)
    assert_sequences([(w, h) for w, h, _ in units], n, sms)
    H, W = bottom + 8, 2112
    frames = make_frames(boxes, n, H, W, 1100)
    (x, y, w, h), _ = boxes[-1]
    rng = np.random.default_rng(5)
    inner = frames[0, y + 10:y + h - 10, x + 10:x + w - 10]
    inner[rng.random(inner.shape) < 0.25] = 255
    insp.configure(Grid(boxes=boxes), is_reference=True)
    rec, _, _, raw = run(insp, frames, vi_b200.default_params(**CONFIG5), K=1024)
    assert rec[0, len(units) - 1]['n_kept'] > 1024
    nk = check_blobs(insp, frames, boxes, CONFIG5, rec, raw, 1024)
    assert nk[0, -1] > 1024


# ---- 6. ragged sequences on the default kernel: no stale slots --------------------------------------------------------

def test_spec_ragged_sequences_leave_no_stale_slots(insp):
    """G1 with salt noise in every other image: some CTA runs a unit with many kept components and next one with few.
    The slots past the second unit's count still hold the sentinel."""
    sms = sm_count()
    n = frames_for(len(G1), sms)
    boxes, _, bottom = shelf_layout(G1, 1008)
    frames = salted(boxes, n, bottom + 8, 1024, 1300, lambda i: 0.05 if i % 2 == 0 else 0.0)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    K = 64
    rec, _, _, raw = run(insp, frames, vi_b200.default_params(**CONFIG5), K=K)
    nk = rec['n_kept'].reshape(-1)
    total = nk.size
    nb = min(total, sms)
    pairs = [(u, u + nb) for u in range(total - nb) if nk[u] >= 20 and 0 < nk[u + nb] <= 5]
    assert pairs, "no CTA runs a many-component unit followed by a few-component one"
    check_blobs(insp, frames, boxes, CONFIG5, rec, raw, K)


# ---- 7. the host call -------------------------------------------------------------------------------------------------

def test_host_call_blobs_equal_the_device_call(insp, monkeypatch):
    """Bytes, packed and records-only formats, six chunks over the three slots: the valid entries equal the device
    call's."""
    boxes, _, bottom = shelf_layout(G1, 1008)
    frames = salted(boxes, 12, bottom + 8, 1024, 1500, lambda i: 0.05 if i % 3 == 0 else 0.0)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    p = vi_b200.default_params(**CONFIG5)
    K = 16
    drec, _, _, draw = run(insp, frames, p, K=K)
    monkeypatch.setenv("VI_HOST_CHUNK", "2")
    for fmt in ("bytes", "packed", "none"):
        hrec, _, _, hblobs = insp.inspect_batch_host(frames, p, mask_format=fmt, max_blobs=K)
        assert hblobs.shape == (12, insp.n_units, K) and hblobs.dtype == vi_b200.BLOB_DTYPE
        assert_records_equal(hrec.reshape(drec.shape), drec, skip=DIAG)
        for fi in range(12):
            for u in range(insp.n_units):
                a = insp.kept_blobs(hrec, hblobs, fi, u)
                b = insp.kept_blobs(drec, draw, fi, u)
                assert a.tobytes() == b.tobytes(), (fmt, fi, u)
    assert drec['n_kept'].max() > K


# ---- 8. arguments -----------------------------------------------------------------------------------------------------

def test_blob_arguments(insp):
    import torch
    boxes = dense_small(3, 2)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    frames = salted(boxes, 2, 320, 448, 1700, lambda i: 0.15)
    tab = torch.full((2 * insp.n_units, 8, 40), SENT, dtype=torch.uint8, device="cuda")
    for k in (0, -1, 1025):
        assert insp._lib.vi_set_defect_blob_output(insp._ctx, C.c_void_p(tab.data_ptr()), k) == -1
    assert insp._lib.vi_set_defect_blob_output(insp._ctx, None, 0) == 0
    rec = np.empty(2 * insp.n_units, vi_b200.RECORD_DTYPE)
    hb = np.empty(2 * insp.n_units * 8, vi_b200.BLOB_DTYPE)
    for k in (0, 1025):
        assert insp._lib.vi_inspect_batch_host_blobs(
            insp._ctx, frames.ctypes.data, 2, 448, 320, 448, 448 * 320, C.byref(vi_b200.default_params()), 2, None, None,
            rec.ctypes.data, hb.ctypes.data, k) == -1
    with pytest.raises(ValueError):
        insp.inspect_batch_host(frames, max_blobs=1025)
    with pytest.raises(ValueError):
        insp.inspect_batch(torch.from_numpy(frames).cuda(), defect_blobs=tab[:1])
    # a table switched on, then off (defect_blobs=None sets NULL): the second batch writes nothing into it
    p = vi_b200.default_params(**CONFIG5)
    rec1, _, _ = insp.inspect_batch(torch.from_numpy(frames).cuda(), p, defect_blobs=tab)
    torch.cuda.synchronize()
    assert (tab != SENT).any()
    tab.fill_(SENT)
    insp.inspect_batch(torch.from_numpy(frames).cuda(), p)
    torch.cuda.synchronize()
    assert (tab == SENT).all()


# ---- 9. the self-checked build ----------------------------------------------------------------------------------------

def test_checked_build_over_blob_tables():
    """Cases 3 and 5 under the self-checked library (VI_CHECKED bounds asserts, the blob slot table's included)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    from vi_b200 import _build
    _build.build(checked=True)
    env = dict(os.environ, VI_B200_LIB="checked")
    res = subprocess.run([sys.executable, os.path.join(root, "tests", "checked_blob_run.py")], env=env,
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "check_word 0" in res.stdout, res.stdout + res.stderr
