"""CUDA path (through the C ABI) against the CPU oracle and the reference goldens.
Run on the B200 box: python -m pytest tests -m gpu"""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

from oracle import ref_cv2 as R
from oracle import restate as S
import vi_b200
from vi_b200 import synth
from vi_b200.grid import Grid, generate_grid


@pytest.fixture(scope="module")
def insp():
    return vi_b200.Inspector(0)


def crops(n=3, seed0=500, shape=(315, 316)):
    h, w = shape
    out = []
    for s in range(n):
        fr = synth.make_frame(seed0 + s, [(8, 8, w, h)], H=h + 16, W=w + 16)
        out.append(fr[8:8 + h, 8:8 + w].copy())
    return out


def adversarial_masks():
    rng = np.random.default_rng(5)
    ms = [np.zeros((17, 23), np.uint8), np.full((17, 23), 255, np.uint8), np.full((1, 1), 255, np.uint8),
          np.zeros((1, 40), np.uint8)]
    m = np.zeros((40, 40), np.uint8); m[5:35, 5:35] = 255; m[10:30, 10:30] = 0; m[15:25, 15:25] = 255; m[18:22, 18:22] = 0
    ms.append(m)
    m = np.zeros((30, 30), np.uint8); np.fill_diagonal(m, 255); ms.append(m)
    m = np.zeros((30, 31), np.uint8); m[::2, ::2] = 255; m[1::2, 1::2] = 255; ms.append(m)
    m = np.zeros((30, 30), np.uint8); m[0, :] = m[-1, :] = 255; m[:, 0] = m[:, -1] = 255; m[10:14, 10:14] = 255; ms.append(m)
    m = np.zeros((33, 35), np.uint8); m[16, :] = 255; m[:, 17] = 255; ms.append(m)
    m = np.zeros((12, 12), np.uint8); m[2:5, 2:5] = 255; m[5:8, 5:8] = 255; ms.append(m)
    m = np.zeros((20, 20), np.uint8); m[4:16, 4:16] = 255; m[6:14, 6:14] = 0; m[9, 4:6] = 0; ms.append(m)
    m = np.zeros((20, 40), np.uint8); m[10:14, 2:6] = 255; m[3:7, 30:34] = 255; ms.append(m)      # area tie
    m = np.zeros((21, 40), np.uint8); m[5:9, 30:34] = 255; m[4:8, 2:6] = 255; m[4, 2] = 0; m[8, 5] = 255; ms.append(m)
    ms.append((rng.random((200, 210)) < 0.02).astype(np.uint8) * 255)
    ms.append((rng.random((150, 160)) < 0.55).astype(np.uint8) * 255)
    ms.append((rng.random((315, 316)) < 0.5).astype(np.uint8) * 255)      # run table overflows shared memory
    ms.append((rng.random((64, 70)) < 0.3).astype(np.uint8) * 7)          # non-255 foreground values
    m = np.zeros((315, 316), np.uint8); m[::2, ::2] = 255; ms.append(m)   # maximal run count
    # spiral: long dependency chains for the union-find
    m = np.zeros((101, 101), np.uint8)
    x = y = 0; dx, dy = 1, 0; n = 101
    lo_x, hi_x, lo_y, hi_y = 0, 100, 0, 100
    while lo_x <= hi_x and lo_y <= hi_y:
        m[lo_y, lo_x:hi_x + 1] = 255; m[lo_y:hi_y + 1, hi_x] = 255
        if hi_y - lo_y >= 2: m[hi_y, lo_x + 2:hi_x + 1] = 255
        if hi_x - lo_x >= 2: m[lo_y + 2:hi_y + 1, lo_x + 2] = 255
        lo_x += 4; lo_y += 4; hi_x -= 4; hi_y -= 4
    ms.append(m)
    return ms


@pytest.mark.parametrize("r", [0, 1, 2, 3, 6, 7, 17, 40, 63, 200])
def test_erode_square(insp, r):
    for m in adversarial_masks() + [R.segment_cell(c) for c in crops(2)]:
        ref = cv2.erode(((m > 0) * 255).astype(np.uint8), None, iterations=r) if r > 0 else ((m > 0) * 255).astype(np.uint8)
        got = insp.erode_square(m, r)
        assert np.array_equal(got, ref), (r, m.shape, int((got != ref).sum()))


def test_fill_internal_holes(insp):
    for m in adversarial_masks():
        ref = R.fill_internal_holes(m)
        got = insp.fill_internal_holes(m)
        assert np.array_equal(got, ref), (m.shape, int((got != ref).sum()))


def test_mask_stats(insp):
    from vi_b200 import segmentation as seg
    for m in adversarial_masks():
        assert seg.mask_stats(m) == R.mask_stats(m)


def test_label_components(insp):
    for m in adversarial_masks():
        res = insp.label_components(m)
        lab_ref, n_ref = S.label8(m)
        assert res["n"] == n_ref
        assert np.array_equal(res["labels"], lab_ref), m.shape
        src = (m > 0).astype(np.uint8)
        nlab, labels, stats, _ = cv2.connectedComponentsWithStats(src, connectivity=8)
        if nlab <= 1:
            assert res["best_label"] == 0 and res["centroid"] is None
            continue
        best = 1 + int(np.argmax(stats[1:, cv2.CC_STAT_AREA]))
        assert np.array_equal(res["labels"] == res["best_label"], labels == best), m.shape
        assert res["best_area"] == int(stats[best, cv2.CC_STAT_AREA])
        assert res["centroid"] == R.largest_component_centroid(m)


SEG_CFGS = [dict(), dict(gaussian_blur=5, morph_kernel=5), dict(gaussian_blur=0, morph_kernel=0),
            dict(gaussian_blur=4, morph_kernel=2), dict(gaussian_blur=7, morph_kernel=7),
            dict(gaussian_blur=31, morph_kernel=9), dict(gaussian_blur=1, morph_kernel=1),
            dict(gaussian_blur=2, morph_kernel=4), dict(method='bogus')]


@pytest.mark.parametrize("ki", range(len(SEG_CFGS)))
def test_segment_cell(insp, ki):
    from vi_b200 import segmentation as seg
    rng = np.random.default_rng(3)
    imgs = crops(3) + [rng.integers(0, 256, size=(64, 97), dtype=np.uint8), np.full((40, 50), 123, np.uint8),
                       np.tile(np.linspace(0, 255, 120).astype(np.uint8), (90, 1)),
                       rng.integers(0, 256, size=(12, 15), dtype=np.uint8), rng.integers(0, 256, size=(1, 1), dtype=np.uint8),
                       rng.integers(0, 256, size=(3, 200), dtype=np.uint8)]
    kw = SEG_CFGS[ki]
    for im in imgs:
        ref = R.segment_cell(im, **kw)
        got = seg.segment_cell(im, **kw)
        assert got.flags.writeable and got.dtype == np.uint8
        if not np.array_equal(got, ref):
            # cv2 itself is not reproducible on every host: on the GPU box's CPU the reference path returns a second mask
            # in ~4 % of calls for the 2x2 ellipse on the 12x15 crop (same Otsu threshold; 40 fresh processes x 50 calls,
            # tools/ history in DESIGN.md section 4).  A repeated-call majority and the cv2-free restatement decide.
            votes = sum(np.array_equal(got, R.segment_cell(im, **kw)) for _ in range(15))
            twin = S.segment_cell(im, gaussian_blur=kw.get('gaussian_blur', 3), morph_kernel=kw.get('morph_kernel', 3))
            assert votes >= 10 and np.array_equal(got, twin), (kw, im.shape, int((got != ref).sum()), votes)


def test_otsu_threshold(insp):
    rng = np.random.default_rng(0)
    for i in range(40):
        if i % 2:
            im = rng.integers(0, 256, size=(40, 50), dtype=np.uint8)
        else:
            a, b = rng.integers(0, 256, size=2)
            im = np.where(rng.random((60, 70)) < rng.random(), a, b).astype(np.uint8)
            im = np.clip(im + rng.normal(0, rng.integers(1, 20), im.shape), 0, 255).astype(np.uint8)
        p = vi_b200.default_params(gaussian_blur=0, morph_kernel=0)
        _, t = insp.segment_cell(im, p, return_threshold=True)
        assert t == R.otsu_threshold(im), i


def test_otsu_threshold_near_ties(insp):
    """Histograms whose between-class variance is flat or tied over many bins: the winner is decided by the
    rounding of OpenCV's serial double recurrence (getThreshVal_Otsu_8u; SURVEY A.3), which the GPU scan reproduces
    -- also where it stops early (bins that cannot hold the maximum are never evaluated).  The checker is OpenCV's
    own C++ scan (IPP dispatch off): on exactly tied histograms (mirror-symmetric ones) the closed-source IPP
    routine the cv2 wheel dispatches to by default breaks the tie differently (tests/test_restate_vs_cv2.py states
    both facts); everywhere else the two agree."""
    import cv2
    rng = np.random.default_rng(11)
    p = vi_b200.default_params(gaussian_blur=0, morph_kernel=0)
    cases = []
    for _ in range(60):                                     # two spikes: every threshold between them ties exactly
        a, b = sorted(rng.integers(0, 256, size=2))
        n = int(rng.integers(1, 4000))
        im = np.full(4200, a, np.uint8); im[:n] = b
        cases.append(im.reshape(60, 70))
    for _ in range(40):                                     # three / four spikes of random weights
        v = np.sort(rng.choice(256, size=int(rng.integers(3, 5)), replace=False))
        w = rng.random(len(v)); w /= w.sum()
        cases.append(rng.choice(v, size=(50, 64), p=w).astype(np.uint8))
    for _ in range(30):                                     # symmetric bimodal: near-ties around the middle
        c = int(rng.integers(40, 216)); d = int(rng.integers(5, 40)); s = float(rng.uniform(0.5, 6))
        half = np.clip(rng.normal(c - d, s, 1600), 0, 255).astype(np.uint8)
        cases.append(np.concatenate([half, (2 * c - half.astype(int)).clip(0, 255).astype(np.uint8)]).reshape(40, 80))
    for _ in range(20):                                     # sparse occupancy, long empty stretches
        v = rng.choice(256, size=int(rng.integers(2, 12)), replace=False)
        cases.append(rng.choice(v, size=(30, 41)).astype(np.uint8))
    cases += [np.full((9, 9), 0, np.uint8), np.full((9, 9), 255, np.uint8), np.arange(256, dtype=np.uint8).reshape(16, 16),
              np.array([[0, 255]], np.uint8), np.array([[7]], np.uint8), np.repeat(np.arange(0, 256, 5, dtype=np.uint8), 7).reshape(-1, 7)]
    from oracle import restate as S
    ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        for i, im in enumerate(cases):
            _, t = insp.segment_cell(im, p, return_threshold=True)
            assert t == R.otsu_threshold(im) == S.otsu_from_hist(np.bincount(im.ravel(), minlength=256)), (i, im.shape)
    finally:
        cv2.ipp.setUseIPP(ipp)


@pytest.mark.parametrize("cfg", [(6, 24, 20), (1, 8, 0), (40, 3, 5), (0, 24, 20), (6, 0, 0), (6, 255, 0), (200, 24, 20),
                                 (3, 12, 1)])
def test_detect_defects(insp, cfg):
    r, thr, mn = cfg
    rng = np.random.default_rng(9)
    excl = [{'shape': 'rect', 'x': 50, 'y': 60, 'w': 70, 'h': 30}, {'shape': 'circle', 'cx': 200, 'cy': 180, 'r': 25}]
    cases = []
    for gray in crops(3, seed0=600):
        seg = R.segment_cell(gray)
        R.apply_exclusions(seg, excl, 2, -3)
        cases.append((gray, seg))
    g = rng.integers(0, 256, size=(96, 96), dtype=np.uint8)
    cases.append((g, np.full((96, 96), 255, np.uint8)))                    # uniform noise: every pixel needs the exact rank count
    g2 = crops(1, seed0=610, shape=(60, 340))[0]
    cases.append((g2, np.full(g2.shape, 255, np.uint8)))                   # wide and short: several 32-cell chunks, one row segment
    g3 = rng.integers(0, 256, size=(12, 15), dtype=np.uint8)
    cases.append((g3, np.full(g3.shape, 255, np.uint8)))                   # smaller than the median window
    p = vi_b200.default_params(threshold=thr, min_area=mn, erode_px=r)
    for gray, seg in cases:
        info = {}
        ref = R.detect_defects(gray, seg, 'threshold', thr, mn, r, info)
        got, rec = insp.detect_defects(gray, seg, p, return_record=True)
        assert (ref is None) == (got is None), (cfg, gray.shape)
        if ref is not None:
            assert np.array_equal(got, ref), (cfg, gray.shape, int((got != ref).sum()))
            assert rec["defect_area"] == int((ref > 0).sum())
            assert rec["n_kept"] == info["n_kept"]
        if 'roi' in info:
            assert rec["roi_area"] == int((info['roi'] > 0).sum())


@pytest.mark.parametrize("cfg", [(6, 24, 20), (1, 8, 0), (0, 3, 0), (6, 100, 5), (17, 255, 0), (6, 0, 0), (3, 12, 1)])
def test_detect_defects_canny(insp, cfg):
    """indexing_ui.py:1536-1539: cv2.Canny inside the ROI, then the same contour filter.  Integer: bit-exact."""
    r, thr, mn = cfg
    rng = np.random.default_rng(19)
    cases = []
    for gray in crops(2, seed0=700):
        cases.append((gray, R.segment_cell(gray)))
    g = rng.integers(0, 256, size=(96, 96), dtype=np.uint8)
    cases.append((g, np.full((96, 96), 255, np.uint8)))                    # noise: tens of thousands of edge runs
    g1 = cv2.GaussianBlur(rng.integers(0, 256, size=(200, 210), dtype=np.uint8), (7, 7), 0)
    cases.append((g1, np.full(g1.shape, 255, np.uint8)))
    g2 = rng.integers(0, 256, size=(315, 316), dtype=np.uint8)
    cases.append((g2, np.full(g2.shape, 255, np.uint8)))                   # run table overflows shared memory
    g3 = rng.integers(0, 256, size=(5, 7), dtype=np.uint8)
    cases.append((g3, np.full(g3.shape, 255, np.uint8)))
    p = vi_b200.default_params(defect_method='canny', threshold=thr, min_area=mn, erode_px=r)
    for gray, seg in cases:
        info = {}
        ref = R.detect_defects(gray, seg, 'canny', thr, mn, r, info)
        got, rec = insp.detect_defects(gray, seg, p, return_record=True)
        assert (ref is None) == (got is None), (cfg, gray.shape)
        if ref is not None:
            assert np.array_equal(got, ref), (cfg, gray.shape, int((got != ref).sum()))
            assert rec["defect_area"] == int((ref > 0).sum())
            assert rec["n_kept"] == info["n_kept"]


def _run_batch(insp, g, fi, params, is_reference, refc, exclusions, host=False, labels=False):
    import torch
    grid = Grid(boxes=g.boxes, exclusions=exclusions, ref_centroids=refc or {})
    insp.configure(grid, is_reference=is_reference)
    frame = g.frame(fi)
    if host:
        rec, seg, dfm = insp.inspect_batch_host(frame[None], params)
        return rec, seg, dfm, None
    d = torch.from_numpy(frame[None]).cuda()
    lab = torch.empty(insp.unit_pixels, dtype=torch.int32, device="cuda") if labels else None
    rec, seg, dfm = insp.inspect_batch(d, params, labels=lab)
    torch.cuda.synchronize()
    rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    return rec, seg.cpu().numpy(), dfm.cpu().numpy(), (lab.cpu().numpy() if labels else None)


ADAPT_CFGS = [dict(), dict(adapt_block=11, adapt_C=-3), dict(adapt_block=3, adapt_C=0), dict(adapt_block=201, adapt_C=10),
              dict(adapt_block=50, adapt_C=5, gaussian_blur=0), dict(adapt_block=21, adapt_C=-50, gaussian_blur=7, morph_kernel=5),
              dict(adapt_block=9, adapt_C=2, morph_kernel=0), dict(adapt_block=2, adapt_C=50)]


def test_segment_cell_adaptive(insp):
    """segmentation.py:83-86.  The adaptive mean is a float32 Gaussian: the north star's +-1 LSB class.  The CUDA path
    follows OpenCV's vector path operation for operation; a pixel can differ only where the float mean lands on a .5
    tie in the columns OpenCV's scalar tail handles.  Stated bound: <= 1e-4 of the pixels of the raw threshold mask
    (blur=0, morph=0 rows below compare it directly); measured: 0."""
    from vi_b200 import segmentation as seg
    rng = np.random.default_rng(31)
    imgs = crops(3) + [rng.integers(0, 256, size=(64, 97), dtype=np.uint8), np.full((40, 50), 123, np.uint8),
                       np.tile(np.linspace(0, 255, 120).astype(np.uint8), (90, 1)),
                       rng.integers(0, 256, size=(12, 15), dtype=np.uint8), rng.integers(0, 256, size=(1, 1), dtype=np.uint8),
                       cv2.GaussianBlur(rng.integers(0, 256, size=(200, 203), dtype=np.uint8), (15, 15), 0)]
    bad = tot = 0
    for kw in ADAPT_CFGS:
        for im in imgs:
            ref = R.segment_cell(im, method='adaptive', **kw)
            got = seg.segment_cell(im, method='adaptive', **kw)
            assert got.shape == ref.shape and got.dtype == np.uint8 and set(np.unique(got)) <= {0, 255}
            bad += int((got != ref).sum()); tot += ref.size
            # the raw adaptive threshold mask, no morphology or hole fill in between
            raw_ref = cv2.adaptiveThreshold(im, 255, cv2.ADAPTIVE_THRESH_GAUSSIAN_C, cv2.THRESH_BINARY_INV,
                                            max(3, kw.get('adapt_block', 51) | 1), kw.get('adapt_C', 10))
            p = vi_b200.default_params(seg_method='adaptive', gaussian_blur=0, morph_kernel=0,
                                       adapt_block=kw.get('adapt_block', 51), adapt_C=kw.get('adapt_C', 10))
            raw_got = insp.segment_cell(im, p)
            raw_ref = R.fill_internal_holes(raw_ref)
            bad += int((raw_got != raw_ref).sum()); tot += raw_ref.size
    print(f"adaptive: {bad} mismatching pixels of {tot}")
    assert bad <= 1e-4 * tot, (bad, tot)


@pytest.mark.parametrize("name", ["config1", "config4", "config5", "blur5_morph5", "adaptive", "canny"])
def test_batch_matches_reference_goldens(insp, golden, name):
    g = golden(name)
    meta = g.meta
    refc = {i: (float(c[0]), float(c[1])) for i, c in enumerate(g.z['ref_centroids']) if not np.isnan(c[0])}
    pk = {k: v for k, v in meta['params'].items()}
    for fi in range(len(meta['seeds'])):
        seg_gold = g.masks(f'f{fi}_seg')
        for r in meta['erode_list']:
            p = vi_b200.default_params(**{**pk, 'erode_px': r})
            rec, seg, dfm, _ = _run_batch(insp, g, fi, p, fi == 0, None if fi == 0 else refc, meta['exclusions'])
            segs = insp.split_masks(seg)
            defs = insp.split_masks(dfm)
            dgold = g.defects(fi, r)
            ng = g.z[f'f{fi}_r{r}_ng']
            area = g.z[f'f{fi}_r{r}_area']
            for i in range(len(g.boxes)):
                assert np.array_equal(segs[i], seg_gold[i]), (name, fi, r, i, 'seg', int((segs[i] != seg_gold[i]).sum()))
                if dgold[i] is None:
                    assert rec[i]['n_kept'] == 0 and not defs[i].any(), (name, fi, r, i)
                else:
                    assert rec[i]['n_kept'] > 0
                    assert np.array_equal(defs[i], dgold[i]), (name, fi, r, i, 'defect', int((defs[i] != dgold[i]).sum()))
                assert rec[i]['defect_area'] == area[i], (name, fi, r, i)
                assert (rec[i]['status'] == vi_b200.STATUS_NG) == bool(ng[i]), (name, fi, r, i)
                assert rec[i]['unit'] == i and rec[i]['image'] == 0
            if fi == 0:
                for i in range(len(g.boxes)):
                    assert rec[i]['cx'] == g.z['ref_centroids'][i][0] and rec[i]['cy'] == g.z['ref_centroids'][i][1]


def test_batch_matches_oracle_records_and_labels(insp, golden):
    """Every record field and the raster-canonical ROI labels against the cv2 oracle."""
    g = golden('config4')
    meta = g.meta
    refc = {i: (float(c[0]), float(c[1])) for i, c in enumerate(g.z['ref_centroids']) if not np.isnan(c[0])}
    p = vi_b200.default_params(erode_px=17)
    rec, seg, dfm, lab = _run_batch(insp, g, 1, p, False, refc, meta['exclusions'], labels=True)
    recs, segs, defs = R.inspect_frame(g.frame(1), g.boxes, R.Params(erode_px=17), meta['exclusions'], refc, False)
    labs = insp.split_masks(lab)
    for i, o in enumerate(recs):
        for k in ('seg_area', 'roi_area', 'defect_area', 'n_kept', 'status', 'dx', 'dy'):
            assert rec[i][k] == o[k], (i, k, rec[i][k], o[k])
        assert rec[i]['cx'] == o['cx'] and rec[i]['cy'] == o['cy']
        gray = g.frame(1)[g.boxes[i][0][1]:g.boxes[i][0][1] + 315, g.boxes[i][0][0]:g.boxes[i][0][0] + 316]
        assert rec[i]['otsu_t'] == R.otsu_threshold(cv2.GaussianBlur(gray, (3, 3), 0))
        er = cv2.erode(((segs[i] > 0) * 255).astype(np.uint8), None, iterations=17)
        lab_ref, _ = S.label8(er)
        assert np.array_equal(labs[i], lab_ref), i


def test_host_batch_equals_device_batch(insp, golden):
    import torch
    g = golden('config1')
    grid = Grid(boxes=g.boxes)
    insp.configure(grid, is_reference=True)
    frames = np.stack([g.frame(0), synth.make_frame(11, [b for b, _ in g.boxes]), synth.make_frame(12, [b for b, _ in g.boxes])])
    rec_h, seg_h, def_h = insp.inspect_batch_host(frames)
    rec_d, seg_d, def_d = insp.inspect_batch(torch.from_numpy(frames).cuda())
    torch.cuda.synchronize()
    rec_d = rec_d.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    assert np.array_equal(seg_h, seg_d.cpu().numpy()) and np.array_equal(def_h, def_d.cpu().numpy())
    for k in vi_b200.RECORD_DTYPE.names:
        a, b = rec_h[k], rec_d[k]
        assert np.array_equal(a, b) or (a.dtype.kind == 'f' and np.array_equal(np.isnan(a), np.isnan(b))), k
    assert list(rec_h['image']) == [i for i in range(3) for _ in range(48)]
    # frames 11 and 12 against the oracle
    for fi in (1, 2):
        recs, segs, defs = R.inspect_frame(frames[fi], g.boxes, R.Params(), (), None, True)
        sm = insp.split_masks(seg_h, fi); dm = insp.split_masks(def_h, fi)
        for i in range(48):
            assert np.array_equal(sm[i], segs[i])
            assert np.array_equal(dm[i], defs[i] if defs[i] is not None else np.zeros_like(dm[i]))
            assert rec_h[fi * 48 + i]['status'] == recs[i]['status']


def _records_equal(a, b):
    for k in vi_b200.RECORD_DTYPE.names:
        x, y = a[k], b[k]
        ok = np.array_equal(x, y) or (x.dtype.kind == 'f' and np.array_equal(np.isnan(x), np.isnan(y)) and
                                      np.array_equal(x[~np.isnan(x)], y[~np.isnan(y)]))
        assert ok, k


@pytest.mark.parametrize("chunk", ["1", "2"])
@pytest.mark.parametrize("pinned", [False, True])
def test_host_batch_multi_chunk(insp, golden, monkeypatch, chunk, pinned):
    """The chunked pipeline of the host-buffer call: slot wrap-around (5 images, 1 or 2 per chunk, 3 slots), the
    chunk-local -> batch-global image index, exclusions and centroid shifts, pinned and pageable frames -- every record
    field and both mask sets against the device-resident call."""
    import torch
    g = golden('config4')
    meta = g.meta
    excl = meta['exclusions']
    refc = {i: (float(c[0]), float(c[1])) for i, c in enumerate(g.z['ref_centroids']) if not np.isnan(c[0])}
    insp.configure(Grid(boxes=g.boxes, exclusions=excl, ref_centroids=refc), is_reference=False)
    boxes = [b for b, _ in g.boxes]
    frames = np.stack([synth.make_frame(900 + i, boxes, H=meta['H'], W=meta['W']) for i in range(5)])
    params = vi_b200.default_params(erode_px=9)
    rec_d, seg_d, def_d = insp.inspect_batch(torch.from_numpy(frames).cuda(), params)
    torch.cuda.synchronize()
    rec_d = rec_d.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    assert (rec_d['dx'] != 0).any() or (rec_d['dy'] != 0).any()
    monkeypatch.setenv("VI_HOST_CHUNK", chunk)
    if pinned:
        ht = torch.empty(frames.shape, dtype=torch.uint8, pin_memory=True)
        ht.numpy()[...] = frames
        hf = ht.numpy()
    else:
        hf = frames
    rec_h, seg_h, def_h = insp.inspect_batch_host(hf, params)
    assert np.array_equal(seg_h, seg_d.cpu().numpy()) and np.array_equal(def_h, def_d.cpu().numpy())
    _records_equal(rec_h, rec_d)
    n_units = len(boxes)
    assert list(rec_h['image']) == [i for i in range(5) for _ in range(n_units)]
    # packed-bit masks and the records-only call carry the same information
    rec_p, seg_p, def_p = insp.inspect_batch_host(hf, params, mask_format="packed")
    _records_equal(rec_p, rec_d)
    for fi in range(5):
        for a, b in zip(insp.unpack_masks(seg_p, fi), insp.split_masks(seg_h, fi)):
            assert np.array_equal(a, b)
        for a, b in zip(insp.unpack_masks(def_p, fi), insp.split_masks(def_h, fi)):
            assert np.array_equal(a, b)
    rec_n, seg_n, def_n = insp.inspect_batch_host(hf, params, mask_format="none")
    assert seg_n is None and def_n is None
    _records_equal(rec_n, rec_d)


def test_packed_mask_output_of_the_device_call(insp, golden):
    import torch
    g = golden('config1')
    insp.configure(Grid(boxes=g.boxes), is_reference=True)
    d = torch.from_numpy(np.stack([g.frame(0), g.frame(0)[::-1].copy()])).cuda()
    sb = torch.zeros(2 * insp.packed_bytes, dtype=torch.uint8, device="cuda")
    db = torch.zeros(2 * insp.packed_bytes, dtype=torch.uint8, device="cuda")
    rec, seg, dfm = insp.inspect_batch(d, seg_bits=sb, defect_bits=db)
    torch.cuda.synchronize()
    seg, dfm, sb, db = seg.cpu().numpy(), dfm.cpu().numpy(), sb.cpu().numpy(), db.cpu().numpy()
    for fi in range(2):
        for a, b in zip(insp.unpack_masks(sb, fi), insp.split_masks(seg, fi)):
            assert np.array_equal(a, b)
        for a, b in zip(insp.unpack_masks(db, fi), insp.split_masks(dfm, fi)):
            assert np.array_equal(a, b)
    # a later call without the packed outputs must not write them
    sb2 = torch.from_numpy(sb.copy()).cuda()
    insp.inspect_batch(d)
    torch.cuda.synchronize()
    assert np.array_equal(sb2.cpu().numpy(), sb)


def test_calls_are_ordered_without_caller_synchronisation(insp, golden):
    """An asynchronous batch followed at once by table updates and blocking per-unit calls of the same context (they run
    on internal streams and share its scratch): the library orders them itself (include/vi_b200.h, Ordering)."""
    import torch
    g = golden('config1')
    boxes = [b for b, _ in g.boxes]
    frames = np.stack([synth.make_frame(700 + i, boxes) for i in range(16)])
    d = torch.from_numpy(frames).cuda()
    crop = crops(1)[0]
    want_seg = R.segment_cell(crop)
    insp.configure(Grid(boxes=g.boxes), is_reference=True)
    ref_rec, ref_seg, ref_def = insp.inspect_batch(d)
    torch.cuda.synchronize()
    ref_rec, ref_seg, ref_def = ref_rec.clone(), ref_seg.clone(), ref_def.clone()
    side = torch.cuda.Stream()
    for rep in range(6):
        rec, seg, dfm = insp.inspect_batch(d)                         # asynchronous, torch's current stream
        got = insp.segment_cell(crop)                                 # internal stream, same scratch slot
        assert np.array_equal(got, want_seg)
        if rep % 2:
            insp.set_grid([b for b in boxes])                         # same tables, rewritten while the batch may run
            with torch.cuda.stream(side):
                rec2, seg2, dfm2 = insp.inspect_batch(d)              # a second stream: ordered after the first
            side.synchronize()
            assert torch.equal(seg2, ref_seg) and torch.equal(rec2, ref_rec)
        torch.cuda.synchronize()
        assert torch.equal(seg, ref_seg) and torch.equal(dfm, ref_def) and torch.equal(rec, ref_rec)


LARGE_UNITS = [(360, 360), (640, 480), (1000, 60), (2048, 1500)]      # 360 x 360: a square just beyond one SM's shared memory


@pytest.mark.parametrize("wh", LARGE_UNITS)
def test_units_beyond_one_sm(insp, wh):
    """Units that do not fit one SM's shared memory run the same phases over a per-CTA arena in global memory
    (DESIGN.md section 2): segment_cell, detect_defects and the batch call, bit-exact against the oracle."""
    import torch
    w, h = wh
    Wf, Hf = ((w + 48 + 15) // 16) * 16, h + 40
    box = (19, 17, w, h)
    inset = max(4, min(24, h // 5))
    fr = synth.make_frame(4000 + w, [box], H=Hf, W=Wf, inset=inset, max_discs=3)
    rng = np.random.default_rng(w)
    for _ in range(6):                                     # more foreign material than the generator's three discs
        cy, cx, r = int(rng.integers(17 + inset + 8, 17 + h - inset - 8)), int(rng.integers(19 + inset + 8, 19 + w - inset - 8)), int(rng.integers(2, 7))
        yy, xx = np.ogrid[cy - r:cy + r + 1, cx - r:cx + r + 1]
        fr[cy - r:cy + r + 1, cx - r:cx + r + 1][(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = int(rng.integers(140, 255))
    crop = fr[17:17 + h, 19:19 + w].copy()
    want_seg = R.segment_cell(crop)
    got_seg, t = insp.segment_cell(crop, return_threshold=True)
    assert t == R.otsu_threshold(cv2.GaussianBlur(crop, (3, 3), 0))
    assert np.array_equal(got_seg, want_seg), int((got_seg != want_seg).sum())
    assert np.array_equal(insp.fill_internal_holes(want_seg), R.fill_internal_holes(want_seg))
    a, sx, sy = insp.mask_sums(want_seg)
    ys, xs = np.nonzero(want_seg)
    assert (a, sx, sy) == (len(xs), int(xs.sum()), int(ys.sum()))
    for r_, thr, mn in ((6, 24, 20), (2, 12, 0)):
        info = {}
        ref = R.detect_defects(crop, want_seg, 'threshold', thr, mn, r_, info)
        got, rec = insp.detect_defects(crop, want_seg, vi_b200.default_params(threshold=thr, min_area=mn, erode_px=r_), return_record=True)
        assert (ref is None) == (got is None)
        if ref is not None:
            assert np.array_equal(got, ref), int((got != ref).sum())
            assert rec["n_kept"] == info["n_kept"] and rec["defect_area"] == int((ref > 0).sum())
        assert rec["roi_area"] == int((info['roi'] > 0).sum())
    # the batch call: two frames, exclusions, centroid shift against the first frame's centroids
    excl = [{'shape': 'rect', 'x': w // 4, 'y': h // 3, 'w': w // 8, 'h': max(3, h // 10)},
            {'shape': 'circle', 'cx': (2 * w) // 3, 'cy': h // 2, 'r': max(3, min(w, h) // 8)}]
    fr2 = np.roll(fr, (2, -3), axis=(0, 1))
    frames = np.stack([fr, fr2])
    recs0, segs0, defs0 = R.inspect_frame(fr, [(box, 0)], R.Params(), excl, None, True)
    refc = {0: (recs0[0]['cx'], recs0[0]['cy'])}
    insp.configure(Grid(boxes=[(box, 0)], exclusions=excl, ref_centroids=refc), is_reference=False)
    rec, seg, dfm = insp.inspect_batch(torch.from_numpy(frames).cuda())
    torch.cuda.synchronize()
    rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    seg, dfm = seg.cpu().numpy(), dfm.cpu().numpy()
    for fi in range(2):
        recs, segs, defs = R.inspect_frame(frames[fi], [(box, 0)], R.Params(), excl, refc, False)
        assert np.array_equal(insp.split_masks(seg, fi)[0], segs[0])
        d = defs[0] if defs[0] is not None else np.zeros((h, w), np.uint8)
        assert np.array_equal(insp.split_masks(dfm, fi)[0], d)
        for k in ('status', 'defect_area', 'seg_area', 'roi_area', 'dx', 'dy', 'n_kept'):
            assert rec[fi][k] == recs[0][k], (fi, k, rec[fi][k], recs[0][k])
    assert (rec[1]['dx'], rec[1]['dy']) != (0, 0)


def test_unit_size_bound_is_documented_and_loud(insp):
    """Beyond the documented bound (4096 wide, 8192 high, 2^24 pixels) the call fails with VI_ERR_TOO_LARGE -- no fallback."""
    with pytest.raises(vi_b200.ViError) as e:
        insp.set_grid([(0, 0, 5000, 100)])
    assert e.value.code == -4
    for rect in ((0, 0, 4096, 4097), (0, 0, 2049, 8192), (0, 0, 4097, 1), (0, 0, 1, 8193)):
        with pytest.raises(vi_b200.ViError) as e:
            insp.set_grid([(0, 0, 8, 8), rect])
        assert e.value.code == -4 and "bound" in str(e.value), rect


def test_config5_full_size_against_the_oracle(insp):
    """BASELINE configs[4] as stated: one 16384x12000 frame, 11,904 units of 96x96 on a 128-pixel lattice, salt noise in
    the plates, threshold 8 / min-area 0 / erode 1 (hundreds of components per unit).  Every record and every mask of
    every unit against the cv2 oracle."""
    import torch
    boxes = synth.dense_grid_boxes()
    assert len(boxes) == 11904
    fr = synth.make_frame(5, boxes, H=12000, W=16384, inset=8, salt_p=0.02)
    p = vi_b200.default_params(threshold=8, min_area=0, erode_px=1)
    bx = [(b, i) for i, b in enumerate(boxes)]
    insp.configure(Grid(boxes=bx), is_reference=True)
    rec, seg, dfm = insp.inspect_batch(torch.from_numpy(fr[None]).cuda(), p)
    torch.cuda.synchronize()
    rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    segs = insp.split_masks(seg.cpu().numpy())
    defs = insp.split_masks(dfm.cpu().numpy())
    recs, osegs, odefs = R.inspect_frame(fr, bx, R.Params(threshold=8, min_area=0, erode_px=1), (), None, True)
    n_kept = 0
    for i in range(len(boxes)):
        assert np.array_equal(segs[i], osegs[i]), (i, 'seg')
        want = odefs[i] if odefs[i] is not None else np.zeros_like(defs[i])
        assert np.array_equal(defs[i], want), (i, 'defect', int((defs[i] != want).sum()))
        for k in ('status', 'defect_area', 'seg_area', 'roi_area', 'n_kept', 'dx', 'dy'):
            assert rec[i][k] == recs[i][k], (i, k, rec[i][k], recs[i][k])
        assert rec[i]['cx'] == recs[i]['cx'] and rec[i]['cy'] == recs[i]['cy']
        n_kept += int(rec[i]['n_kept'])
    assert n_kept > 4 * len(boxes)                        # several kept components per unit (the 3x3 opening removes lone salt pixels)


def test_checked_build_over_adversarial_inputs():
    """The same sources built with -DVI_CHECKED=1 (bounds asserts on the threshold band's list, the run tables and their
    shared / global choice, union-find parents, the dirty-cell and ambiguous-pixel lists, lattice slots, histogram
    counters) over the adversarial masks, noise crops, the default-configuration batch and dense small units: no check
    may fire.  Stands in for compute-sanitizer, which the GPU pool refuses."""
    import subprocess
    import sys
    from vi_b200 import _build
    _build.build(force=False, checked=True)
    env = dict(os.environ, VI_B200_LIB="checked")
    res = subprocess.run([sys.executable, os.path.join(os.path.dirname(__file__), "checked_run.py")], env=env,
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert "check_word 0" in res.stdout, res.stdout[-2000:]
    # and the production library says so when asked for a check word
    import ctypes as C
    insp = vi_b200.Inspector(0)
    w = C.c_uint32(0)
    assert insp._lib.vi_debug_check_word(insp._ctx, C.byref(w)) == -3


def test_full_size_batch_properties(insp, golden):
    """BASELINE configs[1] at its full size (64 frames of 4096x3000, 3,072 units) through size-independent
    properties: the golden frame's units match the reference's outputs wherever the frame sits in the batch; copies of
    a frame give identical records and masks (no state leaks between units or launches); a permuted batch gives the
    permuted result; the host-buffer call equals the device call; NG counts equal the CPU oracle's."""
    import torch
    g = golden('config1')
    boxes = [b for b, _ in g.boxes]
    nu = len(boxes)
    distinct = [g.frame(0)] + [synth.make_frame(s, boxes) for s in (1, 2, 3)]
    order = [int(i) for i in np.random.default_rng(4).integers(0, 4, size=64)]
    order[0], order[63] = 0, 0
    frames = np.stack([distinct[i] for i in order])
    insp.configure(Grid(boxes=g.boxes), is_reference=True)
    d = torch.from_numpy(frames).cuda()
    rec, seg, dfm = insp.inspect_batch(d)
    torch.cuda.synchronize()
    rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(64, nu)
    seg = seg.cpu().numpy().reshape(64, -1)
    dfm = dfm.cpu().numpy().reshape(64, -1)
    first = {}
    for k, i in enumerate(order):
        if i not in first:
            first[i] = k
            continue
        f = first[i]
        for name in ('otsu_t', 'seg_area', 'roi_area', 'defect_area', 'n_kept', 'status', 'dx', 'dy', 'cx', 'cy'):
            assert np.array_equal(rec[k][name], rec[f][name]), (k, name)
        assert np.array_equal(seg[k], seg[f]) and np.array_equal(dfm[k], dfm[f]), k
        assert (rec[k]['image'] == k).all() and (rec[k]['unit'] == np.arange(nu)).all()
    # the golden frame (reference outputs) at both ends of the batch
    seg_gold = g.masks('f0_seg')
    dgold = g.defects(0, 6)
    for k in (0, 63):
        segs = insp.split_masks(seg[k]); defs = insp.split_masks(dfm[k])
        for u in range(nu):
            assert np.array_equal(segs[u], seg_gold[u]), (k, u)
            ref = dgold[u] if dgold[u] is not None else np.zeros_like(defs[u])
            assert np.array_equal(defs[u], ref), (k, u)
    # NG counts of the other frames against the CPU oracle
    for i in (1, 2, 3):
        recs, _, _ = R.inspect_frame(distinct[i], g.boxes, R.Params(), (), None, True)
        assert [int(r['status']) for r in recs] == rec[first[i]]['status'].tolist(), i
    # permutation: reversed batch gives the reversed result
    rec2, seg2, dfm2 = insp.inspect_batch(torch.flip(d, dims=[0]).contiguous())
    torch.cuda.synchronize()
    rec2 = rec2.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(64, nu)
    assert np.array_equal(rec2['status'][::-1], rec['status']) and np.array_equal(rec2['defect_area'][::-1], rec['defect_area'])
    assert np.array_equal(seg2.cpu().numpy().reshape(64, -1)[::-1], seg) and np.array_equal(dfm2.cpu().numpy().reshape(64, -1)[::-1], dfm)
    # host-buffer call
    hrec, hseg, hdef = insp.inspect_batch_host(frames)
    assert np.array_equal(hseg.reshape(64, -1), seg) and np.array_equal(hdef.reshape(64, -1), dfm)
    assert np.array_equal(hrec['status'].reshape(64, nu), rec['status']) and np.array_equal(hrec['image'].reshape(64, nu), rec['image'])


def test_config4_full_size_erosion_sweep(insp):
    """BASELINE configs[3] as stated: the grid.json grid on a full 4096x3000 frame, rectangle + circle exclusions, a
    per-unit centroid shift against a reference frame (grid JSON v2, indexing_ui.py:2296-2338), erosion radii across
    1..63 (direct passes up to 10, window doubling above): every unit's masks and record against the cv2 oracle."""
    import torch
    boxes = generate_grid((251, 232, 316, 315), 4, 6, 2, 1, 133, 136, 252, 0)
    frames = np.stack([synth.make_frame(s, [b for b, _ in boxes]) for s in (40, 41)])
    excl = [{'shape': 'rect', 'x': 50, 'y': 60, 'w': 70, 'h': 30}, {'shape': 'circle', 'cx': 200, 'cy': 180, 'r': 25}]
    recs0, _, _ = R.inspect_frame(frames[0], boxes, R.Params(), excl, None, True)
    refc = {i: (r['cx'], r['cy']) for i, r in enumerate(recs0) if r['cx'] == r['cx']}
    insp.configure(Grid(boxes=boxes, exclusions=excl, ref_centroids=refc), is_reference=False)
    d = torch.from_numpy(frames[1:2]).cuda()
    shifted = 0
    for r in (1, 10, 11, 63):
        rec, seg, dfm = insp.inspect_batch(d, vi_b200.default_params(erode_px=r))
        torch.cuda.synchronize()
        rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
        segs = insp.split_masks(seg.cpu().numpy()); defs = insp.split_masks(dfm.cpu().numpy())
        recs, osegs, odefs = R.inspect_frame(frames[1], boxes, R.Params(erode_px=r), excl, refc, False)
        for u, o in enumerate(recs):
            assert np.array_equal(segs[u], osegs[u]), (r, u, 'seg')
            ref = odefs[u] if odefs[u] is not None else np.zeros_like(defs[u])
            assert np.array_equal(defs[u], ref), (r, u, 'defect')
            for k in ('seg_area', 'roi_area', 'defect_area', 'n_kept', 'status', 'dx', 'dy'):
                assert rec[u][k] == o[k], (r, u, k, rec[u][k], o[k])
            shifted += int(o['dx'] != 0 or o['dy'] != 0)
    assert shifted > 0, "the frames' jitter should shift some centroids"


def test_ragged_grid_and_unaligned_frames(insp):
    """A grid JSON may hold arbitrary boxes (indexing_ui.py:2881-2889): units of different sizes in one batch, on
    frames whose width is not a multiple of 16 (the scalar gather), with exclusions and a centroid shift, against the
    cv2 oracle unit by unit."""
    import torch
    boxes = [((7, 5, 316, 315), 0), ((340, 9, 200, 150), 1), ((560, 20, 96, 96), 2), ((700, 3, 40, 33), 3),
             ((760, 50, 13, 21), 4), ((340, 170, 333, 120), 5), ((800, 100, 150, 230), 6), ((690, 60, 3, 3), 7),
             ((10, 335, 500, 60), 8),        # wide units: the lattice's column pass takes several 32-cell chunks per row segment,
             ((520, 340, 400, 52), 9)]       # more tasks than warps (the Otsu warp takes columns too)
    W, H = 1001, 400
    frames = np.stack([synth.make_frame(s, [b for b, _ in boxes], H=H, W=W, inset=6, jitter=2) for s in (11, 12)])
    excl = [{'shape': 'rect', 'x': 20, 'y': 10, 'w': 30, 'h': 12}, {'shape': 'circle', 'cx': 60, 'cy': 50, 'r': 9}]
    for params in (dict(), dict(erode_px=2, threshold=10, min_area=3)):
        recs0, _, _ = R.inspect_frame(frames[0], boxes, R.Params(**params), excl, None, True)
        refc = {i: (r['cx'], r['cy']) for i, r in enumerate(recs0) if r['cx'] == r['cx']}
        insp.configure(Grid(boxes=boxes, exclusions=excl, ref_centroids=refc), is_reference=False)
        rec, seg, dfm = insp.inspect_batch(torch.from_numpy(frames).cuda(), vi_b200.default_params(**params))
        torch.cuda.synchronize()
        rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(2, len(boxes))
        seg = seg.cpu().numpy().reshape(2, -1); dfm = dfm.cpu().numpy().reshape(2, -1)
        for fi in range(2):
            recs, osegs, odefs = R.inspect_frame(frames[fi], boxes, R.Params(**params), excl, refc, False)
            segs = insp.split_masks(seg[fi]); defs = insp.split_masks(dfm[fi])
            for u, o in enumerate(recs):
                assert np.array_equal(segs[u], osegs[u]), (params, fi, u, 'seg')
                ref = odefs[u] if odefs[u] is not None else np.zeros_like(defs[u])
                assert np.array_equal(defs[u], ref), (params, fi, u, 'defect')
                for k in ('seg_area', 'roi_area', 'defect_area', 'n_kept', 'status', 'dx', 'dy'):
                    assert rec[fi, u][k] == o[k], (params, fi, u, k, rec[fi, u][k], o[k])


def test_async_gather_variants_agree(insp):
    """The default kernel fetches the next unit's crop asynchronously and undoes the crop's byte phase (x0 & 15)
    afterwards: as tensor-map boxes (cp.async.bulk.tensor) when the box tiles of the grid's largest unit fit the staging
    area (gray crop + first mask), else as one bulk copy per row.  Units at every byte phase, on 16-byte aligned frames,
    against the cv2 oracle, one grid per variant:
    boxes: units of several sizes up to 316 x 315 (3 frames: every unit is the first of its CTA, fetched as boxes);
    rows:  16 units of 150 x 230 -- the boxes need 176 B x 232 rows = 40,832 B, more than the 40,496 B of gray + mask,
           the row copies at most 176 x 230 = 40,480 B.  20 frames, so that every CTA (one per SM) fetches later units."""
    import torch
    boxes_grid = [((3 + 37 * i + (i % 16), 8 + 5 * (i % 3), 36, 40), i) for i in range(16)]          # x0 & 15 takes many values
    boxes_grid += [((16, 70, 316, 315), 16), ((349, 72, 316, 315), 17), ((680, 75, 300, 200), 18), ((683, 290, 97, 111), 19)]
    rows_grid = [((16 + 176 * j + 8 * r + j, 8 + 246 * r, 150, 230), 8 * r + j) for r in range(2) for j in range(8)]  # x0 & 15 = 0..15
    for boxes, W, H, seeds in ((boxes_grid, 1024, 420, (31, 32, 33)), (rows_grid, 1424, 496, range(40, 60))):
        frames = np.stack([synth.make_frame(s, [b for b, _ in boxes], H=H, W=W, inset=5, jitter=2) for s in seeds])
        n = len(frames)
        insp.configure(Grid(boxes=boxes), is_reference=True)
        rec, seg, dfm = insp.inspect_batch(torch.from_numpy(frames).cuda())
        torch.cuda.synchronize()
        rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(n, len(boxes))
        seg = seg.cpu().numpy().reshape(n, -1); dfm = dfm.cpu().numpy().reshape(n, -1)
        for fi in range(n):
            recs, osegs, odefs = R.inspect_frame(frames[fi], boxes, R.Params(), (), None, True)
            segs = insp.split_masks(seg[fi]); defs = insp.split_masks(dfm[fi])
            for u, o in enumerate(recs):
                (x, y, w, h), _ = boxes[u]
                otsu = R.otsu_threshold(cv2.GaussianBlur(frames[fi, y:y + h, x:x + w], (3, 3), 0))
                assert rec[fi, u]['otsu_t'] == otsu, (W, fi, u, 'otsu_t')
                assert np.array_equal(segs[u], osegs[u]), (W, fi, u, 'seg')
                ref = odefs[u] if odefs[u] is not None else np.zeros_like(defs[u])
                assert np.array_equal(defs[u], ref), (W, fi, u, 'defect')
                for k in ('seg_area', 'roi_area', 'defect_area', 'n_kept', 'status'):
                    assert rec[fi, u][k] == o[k], (W, fi, u, k)


def test_detect_defects_on_a_bright_region(insp):
    """detect_defects takes any mask (indexing_ui.py:1486-1490).  The median stage brackets the median with levels
    around ONE class of the crop -- the dark one for the path's own inverse-threshold masks, the bright one when the
    caller's mask lives there (one gray sample per mask word votes).  Either choice is exact; this pins the second."""
    rng = np.random.default_rng(77)
    for shape in ((120, 150), (315, 316)):
        h, w = shape
        gray = np.clip(60 + rng.normal(0, 5, size=shape), 0, 255).astype(np.uint8)
        gray[15:h - 15, 15:w - 15] = np.clip(200 + rng.normal(0, 6, size=(h - 30, w - 30)), 0, 255).astype(np.uint8)
        for _ in range(4):                                               # dark specks on the bright plate
            cy, cx = int(rng.integers(30, h - 30)), int(rng.integers(30, w - 30))
            gray[cy - 3:cy + 4, cx - 3:cx + 4] = 90
        seg = np.zeros(shape, np.uint8); seg[15:h - 15, 15:w - 15] = 255
        for (r, thr, mn) in ((6, 24, 20), (2, 10, 3)):
            info = {}
            ref = R.detect_defects(gray, seg, 'threshold', thr, mn, r, info)
            got, rec = insp.detect_defects(gray, seg, vi_b200.default_params(threshold=thr, min_area=mn, erode_px=r), return_record=True)
            assert (ref is None) == (got is None)
            assert ref is not None and (ref > 0).any()
            assert np.array_equal(got, ref), (shape, r, thr, int((got != ref).sum()))
            assert rec["n_kept"] == info["n_kept"]
            if (r, thr) == (6, 24):
                assert rec["n_ambiguous"] < 0.2 * (h * w), "the levels did not follow the mask's class"


def test_seg_stats_output_matches_mask_stats(insp, golden, tmp_path):
    """The optional per-unit (area, sum x, sum y) of the final seg masks (SURVEY n4) against the reference's
    mask_stats on the masks themselves, and the CSV rows built from it against rows built the reference's way."""
    import csv
    import torch
    from vi_b200 import export
    g = golden('config4')
    meta = g.meta
    refc = {i: (float(c[0]), float(c[1])) for i, c in enumerate(g.z['ref_centroids']) if not np.isnan(c[0])}
    insp.configure(Grid(boxes=g.boxes, exclusions=meta['exclusions'], ref_centroids=refc), is_reference=False)
    d = torch.from_numpy(g.frame(1)[None]).cuda()
    stats = torch.full((len(g.boxes), 3), -1, dtype=torch.int64, device='cuda')
    rec, seg, _ = insp.inspect_batch(d, seg_stats=stats)
    torch.cuda.synchronize()
    segs = insp.split_masks(seg.cpu().numpy())
    rows = export.masks_summary_rows(stats.cpu().numpy())
    rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    for i, m in enumerate(segs):
        st = R.mask_stats(m)
        assert rows[i]['area'] == st['area'] == rec[i]['seg_area']
        assert (rows[i]['centroid_x'], rows[i]['centroid_y']) == st['centroid'], i
    export.write_masks_summary_csv(str(tmp_path / 'a.csv'), rows)
    with open(tmp_path / 'b.csv', 'w', newline='') as cf:                    # indexing_ui.py:2723-2729 on mask_stats rows
        w = csv.DictWriter(cf, fieldnames=['index', 'mask', 'area', 'centroid_x', 'centroid_y'])
        w.writeheader()
        for i, m in enumerate(segs):
            st = R.mask_stats(m)
            w.writerow({'index': i, 'mask': f'mask_{i:04d}.png', 'area': st['area'], 'centroid_x': st['centroid'][0], 'centroid_y': st['centroid'][1]})
    assert (tmp_path / 'a.csv').read_bytes() == (tmp_path / 'b.csv').read_bytes()
    # switched off again: the buffer stays untouched
    stats.fill_(-7)
    insp.inspect_batch(d)
    torch.cuda.synchronize()
    assert (stats == -7).all()


def test_randomized_parameters_against_oracle(insp):
    """Seeded sweep over the widget ranges (threshold, erosion radius, min-area, blur and morphology sizes, both
    segmentation and defect methods) on frames of varying contrast, noise and plate geometry: every unit's masks and
    record against the cv2 oracle."""
    import torch
    rng = np.random.default_rng(2024)
    boxes = [((5, 4, 150, 141), 0), ((170, 9, 97, 120), 1), ((280, 2, 64, 64), 2), ((360, 6, 201, 150), 3)]
    W, H = 576, 160
    for trial in range(36):
        params = dict(threshold=int(rng.integers(0, 70)), erode_px=int(rng.integers(0, 24)), min_area=int(rng.integers(0, 60)),
                      gaussian_blur=int(rng.choice([0, 3, 3, 5, 6])), morph_kernel=int(rng.choice([0, 3, 3, 5, 7])))
        if trial % 6 == 4:
            params['defect_method'] = 'canny'
        if trial % 9 == 7:
            params.update(seg_method='adaptive', adapt_block=int(rng.choice([11, 31, 51])), adapt_C=int(rng.integers(2, 15)))
        fr = synth.make_frame(1000 + trial, [b for b, _ in boxes], H=H, W=W, inset=int(rng.integers(4, 20)), jitter=2,
                              max_discs=int(rng.integers(0, 6)), salt_p=float(rng.choice([0.0, 0.0, 0.01, 0.05])))
        if trial % 5 == 3:                                   # low contrast: classes close together
            fr = (fr.astype(np.int32) // 3 + 80).astype(np.uint8)
        rp = R.Params(**{k: (v if not isinstance(v, str) else v) for k, v in params.items()})
        recs, osegs, odefs = R.inspect_frame(fr, boxes, rp, (), None, True)
        insp.configure(Grid(boxes=boxes), is_reference=True)
        rec, seg, dfm = insp.inspect_batch(torch.from_numpy(fr[None]).cuda(), vi_b200.default_params(**params))
        torch.cuda.synchronize()
        rec = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
        segs = insp.split_masks(seg.cpu().numpy()); defs = insp.split_masks(dfm.cpu().numpy())
        for u, o in enumerate(recs):
            assert np.array_equal(segs[u], osegs[u]), (trial, params, u, 'seg', int((segs[u] != osegs[u]).sum()))
            ref = odefs[u] if odefs[u] is not None else np.zeros_like(defs[u])
            assert np.array_equal(defs[u], ref), (trial, params, u, 'defect', int((defs[u] != ref).sum()))
            for k in ('seg_area', 'roi_area', 'defect_area', 'n_kept', 'status'):
                assert rec[u][k] == o[k], (trial, params, u, k, rec[u][k], o[k])


def test_frame_ingest(insp):
    """Device ingest (SURVEY n3) against the reference's host calls: aligned frames (vector kernels) and odd
    shapes / pitches (scalar kernels), batch of frames, mono identity."""
    import torch
    rng = np.random.default_rng(9)
    for n, H, W in ((3, 64, 4096), (2, 37, 131), (1, 5, 16), (1, 1, 1)):
        a = rng.integers(0, 256, size=(n, H, W, 4), dtype=np.uint8)
        if W >= 16:
            a[0, 0, :8] = [[v, v, v, 255] for v in (0, 1, 127, 128, 254, 255, 17, 200)]
        got = insp.ingest_argb32(torch.from_numpy(a).cuda()).cpu().numpy()
        for i in range(n):
            assert np.array_equal(got[i], R.gray_from_argb32(a[i])), (n, H, W, i)
        u = rng.integers(0, 65536, size=(n, H, W), dtype=np.uint16)
        got = insp.ingest_gray16(torch.from_numpy(u.view(np.int16)).cuda()).cpu().numpy()
        assert np.array_equal(got, R.gray8_from_gray16(u)), (n, H, W)
    # a view with a row pitch wider than the frame (unaligned start: scalar kernel)
    big = rng.integers(0, 256, size=(2, 40, 200, 4), dtype=np.uint8)
    view = torch.from_numpy(big).cuda()[:, 3:35, 5:165]
    got = insp.ingest_argb32(view).cpu().numpy()
    for i in range(2):
        assert np.array_equal(got[i], R.gray_from_argb32(big[i, 3:35, 5:165]))


def test_fast_division_is_ieee(insp):
    """The Otsu recurrence divides through a precomputed reciprocal (two residual
    corrections); it must be the correctly rounded quotient, bit for bit."""
    import ctypes as C
    from vi_b200 import _lib
    bad = C.c_int64(-1)
    _lib.check(insp._lib.vi_debug_fastdiv_check(insp._ctx, 1 << 28, 12345, C.byref(bad)))
    assert bad.value == 0


def test_error_paths(insp):
    from vi_b200 import segmentation as seg
    assert seg.fill_internal_holes(None) is None
    with pytest.raises(ValueError):
        seg.fill_internal_holes(np.zeros((2, 2, 2), np.uint8))
    assert seg.mask_stats(np.zeros((4, 4), np.uint8)) == {'area': 0, 'centroid': (0, 0)}
    with pytest.raises(vi_b200.ViError):
        insp.segment_cell(np.zeros((8, 8), np.uint8), vi_b200.default_params(seg_method=7))             # not a reference option
    with pytest.raises(vi_b200.ViError):
        insp.segment_cell(np.zeros((8, 8), np.uint8), vi_b200.default_params(median_ksize=5))           # the reference hard-codes 21
    insp.set_grid([(0, 0, 2000, 2000)])                                      # beyond one SM's shared memory: the arena path takes it
    with pytest.raises(vi_b200.ViError):
        insp.set_grid([(0, 0, 4097, 100)])                                   # beyond the documented bound of a unit
    insp.set_grid([(10, 10, 50, 50)])
    import torch
    with pytest.raises(vi_b200.ViError):
        insp.inspect_batch(torch.zeros((1, 40, 40), dtype=torch.uint8, device='cuda'))   # rect leaves the frame
