"""Runs the CUDA path of the self-checked library (libvi_b200_checked.so: -DVI_CHECKED=1, bounds asserts on every list
and table with a capacity) over adversarial and ordinary inputs and prints the check word (0 = no bound was violated).
Started by tests/test_gpu_parity.py::test_checked_build_over_adversarial_inputs with VI_B200_LIB=checked."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
assert os.environ.get("VI_B200_LIB") == "checked"

import torch  # noqa: E402
import vi_b200  # noqa: E402
from vi_b200 import _lib, synth  # noqa: E402
from vi_b200.grid import Grid  # noqa: E402
from test_gpu_parity import adversarial_masks  # noqa: E402
from test_gpu_unit_sequences import ARENA_UNITS, EXCL, G1, G2, frames_for, make_frames, shelf_layout  # noqa: E402


def main():
    insp = vi_b200.Inspector(0)
    rng = np.random.default_rng(1)
    for m in adversarial_masks():
        insp.fill_internal_holes(m)
        insp.label_components(m)
        insp.erode_square(m, 3)
        g = rng.integers(0, 256, size=m.shape, dtype=np.uint8)
        insp.detect_defects(g, np.where(m > 0, 255, 0).astype(np.uint8), vi_b200.default_params(threshold=5, min_area=0, erode_px=0))
        insp.detect_defects(g, np.full(m.shape, 255, np.uint8), vi_b200.default_params(defect_method=1, threshold=30, erode_px=1))
    for shape in ((315, 316), (96, 96), (12, 15), (60, 340), (480, 640)):
        g = rng.integers(0, 256, size=shape, dtype=np.uint8)
        for kw in (dict(), dict(gaussian_blur=5, morph_kernel=5), dict(seg_method=1, adapt_block=11), dict(gaussian_blur=0, morph_kernel=0)):
            insp.segment_cell(g, vi_b200.default_params(**kw))
        insp.detect_defects(g, np.full(shape, 255, np.uint8), vi_b200.default_params(threshold=2, min_area=0, erode_px=1))
    # the default-configuration kernel (asynchronous gather and all): three frames of the grid.json grid
    boxes = vi_b200.generate_grid((251, 232, 316, 315), 4, 6, 2, 1, 133, 136, 252, 0)
    frames = np.stack([synth.make_frame(40 + i, [b for b, _ in boxes]) for i in range(3)])
    frames[2] = rng.integers(0, 256, size=frames[2].shape, dtype=np.uint8)           # pure noise: every list at its worst
    insp.configure(Grid(boxes=boxes, exclusions=[{'shape': 'circle', 'cx': 150, 'cy': 150, 'r': 40}]), is_reference=True)
    for thr in (24, 3):
        insp.inspect_batch(torch.from_numpy(frames).cuda(), vi_b200.default_params(threshold=thr, min_area=0, erode_px=2))
    insp.inspect_batch_host(frames, vi_b200.default_params())
    # dense small units with salt noise (BASELINE configs[4] in miniature)
    small = [(32 + 128 * i, 32 + 128 * j, 96, 96) for j in range(4) for i in range(6)]
    fr = synth.make_frame(9, small, H=576, W=832, inset=8, salt_p=0.02)
    insp.configure(Grid(boxes=[(b, i) for i, b in enumerate(small)]), is_reference=True)
    insp.inspect_batch(torch.from_numpy(fr[None]).cuda(), vi_b200.default_params(threshold=8, min_area=0, erode_px=1))
    # ragged grids, many units of different sizes per CTA: the tensor-box gather (G1), the row-copy gather (G2), the
    # general kernel (G1, blur 5 / morph 5) and the global arena (G1 plus a 640 x 480 unit)
    for units, kws in ((G1, (dict(), dict(gaussian_blur=5, morph_kernel=5))), (G2, (dict(),)),
                       (ARENA_UNITS, (dict(), dict(defect_method=1), dict(seg_method=1, adapt_block=11, adapt_C=5)))):
        boxes, _, bottom = shelf_layout(units, 1008)
        n = frames_for(len(units), torch.cuda.get_device_properties(0).multi_processor_count)
        fr = make_frames(boxes, n, bottom + 8, 1024, 50)
        insp.configure(Grid(boxes=boxes, exclusions=EXCL), is_reference=True)
        for kw in kws:
            insp.inspect_batch(torch.from_numpy(fr).cuda(), vi_b200.default_params(**kw))
    # the device Otsu on its own: adversarial histograms, two with a bad pixel count (VI_ERR_ARG, rows of -1)
    import otsu_families as F
    H, _ = F.mixed(rng, 500)
    npix = H.sum(1)
    npix[:2] = (0, (1 << 24) + 1)
    out = torch.empty((len(H), 3), dtype=torch.int32, device="cuda")
    dh = torch.from_numpy(H.astype(np.uint32).view(np.int32)).cuda()
    dn = torch.from_numpy(npix.astype(np.int32)).cuda()
    assert insp._lib.vi_debug_otsu(insp._ctx, dh.data_ptr(), dn.data_ptr(), len(H), out.data_ptr()) == _lib.VI_ERR_ARG
    torch.cuda.synchronize()
    # the median residual stage on its own with its lists capped (every overflow path), and a batch of noisy plates
    # whose units list from a few to more than 16,384 ambiguous pixels and more than 4,096 dirty cells
    import test_gpu_median_residual as M
    for (h, w) in ((315, 316), (48, 97), (24, 1500), (1, 4096)):
        g = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
        roi = rng.random((h, w)) < 0.7
        for ccap, ecap in ((4096, 16384), (0, 0), (1, 193), (7, 1), (4096, 192)):
            _lib.check(M.stage(insp, g, roi, [100, 128, 156], 3, ccap, ecap)[0])
    boxes, _, bottom = shelf_layout([(w, h, ph) for w, h, _, ph in M.UNITS], 1008)
    fr = M.noisy_frames(boxes, [s for _, _, s, _ in M.UNITS], 3, bottom + 8, 1024, 500)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    insp.inspect_batch(torch.from_numpy(fr).cuda(), vi_b200.default_params(threshold=6))
    torch.cuda.synchronize()
    word = C.c_uint32(12345)
    _lib.check(insp._lib.vi_debug_check_word(insp._ctx, C.byref(word)))
    print("check_word", int(word.value))


if __name__ == "__main__":
    main()
