"""CPU tests of the host side: grid generation / grid JSON v2 semantics against the
reference's (through the cv2 oracle, itself pinned by the goldens), the C-ABI
library's exports, and the header/binding agreement.  No compute calls."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

import vi_b200
from oracle import ref_cv2 as R
from vi_b200 import _lib, grid as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "vi_b200.h")).read()
    declared = set(re.findall(r"\b(vi_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"vi_excl", "vi_params", "vi_unit_record", "vi_ctx"}
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} is declared in include/vi_b200.h but not exported"
    assert set(_lib.EXPORTS) == declared


def test_struct_layouts_match_the_header():
    assert C.sizeof(_lib.ViParams) == 48
    assert C.sizeof(_lib.ViExcl) == 20
    assert _lib.RECORD_DTYPE.itemsize == 64
    assert _lib.RECORD_DTYPE.fields['cx'][1] == 40 and _lib.RECORD_DTYPE.fields['n_ambiguous'][1] == 56
    p = vi_b200.default_params()
    assert (p.seg_method, p.gaussian_blur, p.morph_kernel, p.adapt_block, p.adapt_C) == (0, 3, 3, 51, 10)
    assert (p.defect_method, p.threshold, p.min_area, p.erode_px, p.median_ksize, p.max_area_frac) == (0, 24, 20, 6, 21, 0.98)


def test_adaptive_taps_host_function_matches_cv2():
    """Host-only export: float32 taps of the adaptive mean, bit-equal to cv2 for the widget range 3..201."""
    cv2 = pytest.importorskip("cv2")
    lib = _lib.load()
    for bs in range(3, 202, 2):
        out = np.zeros(bs, np.float32)
        assert lib.vi_debug_adaptive_taps(bs, out.ctypes.data) == 0
        assert np.array_equal(out, cv2.getGaussianKernel(bs, 0, cv2.CV_32F).ravel()), bs
    assert lib.vi_debug_adaptive_taps(4, np.zeros(4, np.float32).ctypes.data) != 0


def test_compute_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(vi_b200.ViError):
        vi_b200.Inspector(0)


def test_generate_grid_matches_reference_rule(golden):
    g = golden('config1')
    assert G.generate_grid((251, 232, 316, 315), 4, 6, 2, 1, 133, 136, 252, 0) == g.boxes
    for args in [((5, 7, 30, 20), 3, 2, 2, 2, 4, 5, 6, 7), ((0, 0, 10, 10), 1, 1, 1, 1, 0, 0, 0, 0),
                 ((1, 2, 3, 4), 0, 5, 1, 1, 0, 0, 0, 0)]:
        assert G.generate_grid(*args) == R.generate_grid(*args)


def test_grid_json_roundtrip_and_legacy_forms(tmp_path):
    boxes = G.generate_grid((10, 20, 30, 40), 2, 2, 1, 1, 5, 6, 0, 0)
    grid = G.Grid(boxes=boxes, exclusions=[{'shape': 'rect', 'x': 1, 'y': 2, 'w': 3, 'h': 4}, {'shape': 'circle', 'cx': 5, 'cy': 6, 'r': 7}],
                  ref_centroids={0: (1.5, 2.25), 3: (7.0, 8.0)}, metadata={'units_x': 2})
    p = tmp_path / "g.json"
    G.save_grid(p, grid)
    raw = json.load(open(p))
    assert raw['version'] == 2 and raw['exclusion_alignment']['type'] == 'seg_centroid_xy'
    assert raw['exclusion_alignment']['ref_centroids']['3'] == {'cx': 7.0, 'cy': 8.0}
    back = G.load_grid(p)
    assert back.boxes == boxes and back.exclusions == grid.exclusions and back.ref_centroids == grid.ref_centroids
    ref = R.load_grid_json(str(p))          # the oracle's restatement of import_grid reads our file the same way
    assert ref['boxes'] == boxes and ref['ref_centroids'] == grid.ref_centroids and ref['exclusions'] == grid.exclusions
    # legacy: bare list, boxes without index, malformed boxes skipped, wrong alignment type ignored
    legacy = [{'x': 1, 'y': 2, 'w': 3, 'h': 4}, {'x': 'bad'}, {'index': 9, 'x': 5, 'y': 6, 'w': 7, 'h': 8}]
    for parsed in (G.parse_grid(legacy), G.parse_grid({'boxes': legacy, 'exclusion_alignment': {'type': 'other', 'ref_centroids': {'0': {'cx': 1, 'cy': 2}}}})):
        assert parsed.boxes == [((1, 2, 3, 4), 0), ((5, 6, 7, 8), 9)]
        assert parsed.ref_centroids == {}
    assert G.parse_grid(42).boxes == []
    r = R.load_grid_json(legacy)
    assert r['boxes'] == G.parse_grid(legacy).boxes


def test_reference_grid_json_parses_like_the_reference(golden):
    g = golden('config1')
    ours = G.parse_grid({'boxes': [{'index': i, 'x': r[0], 'y': r[1], 'w': r[2], 'h': r[3]} for r, i in g.boxes]})
    assert ours.boxes == g.boxes and ours.exclusions == [] and ours.ref_centroids == {}


def test_exclusion_table():
    rows = G.exclusions_to_table([{'shape': 'rect', 'x': 1, 'y': 2, 'w': 3, 'h': 4}, {'shape': 'circle', 'cx': 5, 'cy': 6, 'r': 7},
                                  {'shape': 'blob', 'cx': 1}, {'shape': 'rect', 'x': 'oops'}])
    assert rows == [(0, 1, 2, 3, 4), (1, 5, 6, 7, 0), (1, 1, 0, 0, 0)]


class _FakeBits(bytearray):
    """Stands in for the sip.voidptr QImage.bits() returns: a buffer with setsize()."""
    def setsize(self, n):
        assert n == len(self)


class _FakeQImage:
    class Format:
        Format_ARGB32 = 5

    def __init__(self, bgra):
        self._a = np.ascontiguousarray(bgra, np.uint8)

    def convertToFormat(self, fmt):
        assert fmt == _FakeQImage.Format.Format_ARGB32
        return self

    def bits(self):
        return _FakeBits(self._a.tobytes())

    def sizeInBytes(self):
        return self._a.size

    def height(self):
        return self._a.shape[0]

    def width(self):
        return self._a.shape[1]


def test_qimage_to_gray_array_on_colour_input(monkeypatch):
    """The drop-in's qimage_to_gray_array (a numpy formula) against the reference's rule (segmentation.py:10-24:
    reversed channels into cv2.cvtColor(BGR2GRAY)), computed with cv2 directly, on colour pixels driven through a
    numpy-backed QImage stand-in."""
    cv2 = pytest.importorskip("cv2")
    from vi_b200 import segmentation as seg
    rng = np.random.default_rng(3)
    bgra = rng.integers(0, 256, size=(37, 53, 4), dtype=np.uint8)
    bgra[:8, :, 0] = bgra[:8, :, 1] = bgra[:8, :, 2] = np.arange(53, dtype=np.uint8)[None, :] * 4      # a mono strip: identity
    monkeypatch.setattr(seg, "QImage", _FakeQImage)
    got = seg.qimage_to_gray_array(_FakeQImage(bgra))
    want = cv2.cvtColor(np.ascontiguousarray(bgra[:, :, :3][:, :, ::-1]), cv2.COLOR_BGR2GRAY)
    assert got.dtype == np.uint8 and np.array_equal(got, want)
    assert np.array_equal(got[:8], bgra[:8, :, 0])
    monkeypatch.setattr(seg, "QImage", None)
    with pytest.raises(RuntimeError):
        seg.qimage_to_gray_array(_FakeQImage(bgra))


def test_packed_mask_png_round_trip(tmp_path):
    """The kernel's packed-bit mask layout (rows of 32-bit words, PNG bit order) written as a 1-bit PNG reads back as
    the 0/255 mask: the consumer contract of export_masks_and_csv (indexing_ui.py:2703-2722) on packed output."""
    cv2 = pytest.importorskip("cv2")
    from vi_b200 import export
    rng = np.random.default_rng(2)
    for (h, w) in ((315, 316), (17, 33), (5, 8), (40, 1)):
        mask = (rng.random((h, w)) < 0.4).astype(np.uint8) * 255
        wpr = (w + 31) // 32
        bits = np.zeros((h, wpr * 32), np.uint8)
        bits[:, :w] = mask > 0
        packed = np.packbits(bits, axis=1)                   # big bit order within bytes = VI_MASKS_PACKED
        assert packed.shape == (h, wpr * 4)
        fn = str(tmp_path / f"m_{h}_{w}.png")
        export.write_mask_png(fn, packed, w, h)
        back = cv2.imread(fn, cv2.IMREAD_GRAYSCALE)
        assert back is not None and back.shape == (h, w) and np.array_equal(back, mask)
