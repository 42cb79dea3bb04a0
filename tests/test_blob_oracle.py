"""The kept-defect-component oracle (tests/blob_oracle.py) against itself and cv2, on synthetic units; no GPU."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from oracle import ref_cv2 as R
import vi_b200
from vi_b200 import synth

import blob_oracle as BO


def test_blob_dtype_is_the_c_struct():
    assert vi_b200.BLOB_DTYPE.itemsize == 40
    assert vi_b200.BLOB_DTYPE.names == BO.BLOB_FIELDS
    assert [vi_b200.BLOB_DTYPE.fields[f][1] for f in BO.BLOB_FIELDS] == [0, 4, 8, 12, 16, 20, 24, 32]


CASES = [
    # (unit w, h, frame kwargs, oracle parameters)
    (316, 315, dict(inset=24, max_discs=6), R.Params()),
    (96, 96, dict(inset=8, salt_p=0.02), R.Params(threshold=8, min_area=0, erode_px=1)),
    (96, 96, dict(inset=8, salt_p=0.15), R.Params(threshold=8, min_area=0, erode_px=1)),
    (200, 150, dict(inset=10, max_discs=6), R.Params(defect_method='canny')),
]


@pytest.mark.parametrize("ci", range(len(CASES)))
def test_kept_blobs_partition_the_defect_mask(ci):
    w, h, fkw, rp = CASES[ci]
    seen = 0
    for seed in range(6):
        gray = synth.make_frame(300 + seed, [(0, 0, w, h)], H=h, W=w, jitter=2, **fkw)
        seg, _, _, _ = R.segment_unit(gray, rp)
        info = {}
        dm = R.detect_defects(gray, seg, rp.defect_method, rp.threshold, rp.min_area, rp.erode_px, info)
        kept = BO.kept_contours(gray, seg, **BO.params_kw(rp))
        blobs = BO.describe(kept, gray.shape)
        assert len(blobs) == info.get('n_kept', 0)
        if dm is None:
            assert blobs == []
            continue
        seen += len(blobs)
        assert sum(b['area'] for b in blobs) == int((dm > 0).sum())
        allpix = np.concatenate([b['pixels'] for b in blobs])
        assert np.unique(allpix).size == allpix.size                          # disjoint
        assert np.array_equal(np.sort(allpix), np.flatnonzero(dm.reshape(-1)))  # and together the drawn mask
        firsts = [int(b['pixels'][0]) for b in blobs]
        assert firsts == sorted(firsts)
        for b in blobs:
            assert (b['x'], b['y'], b['w'], b['h']) == cv2.boundingRect(b['contour'])
            full = np.zeros(gray.shape, np.uint8)
            cv2.drawContours(full, [b['contour']], -1, 255, -1)
            assert np.array_equal(np.flatnonzero(full.reshape(-1)), b['pixels'])
            assert b['area2'] == int(2 * cv2.contourArea(b['contour']))
            ys, xs = np.divmod(b['pixels'], w)
            assert b['cx'] == xs.sum() / xs.size and b['cy'] == ys.sum() / ys.size
    assert seen > 0
