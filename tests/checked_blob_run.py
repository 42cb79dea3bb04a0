"""Runs the kept-defect-component table under the self-checked library (libvi_b200_checked.so) and prints the check word
(0 = no bound was violated): dense salted 96 x 96 units at K = 1, 8 and 1024 (shared and global-scratch accumulators)
and the arena kernel over ragged sequences with a 2048 x 1500 unit of more than 1024 components.  Started by
tests/test_gpu_defect_blobs.py::test_checked_build_over_blob_tables with VI_B200_LIB=checked."""
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
from test_gpu_unit_sequences import ARENA_UNITS, frames_for, make_frames, shelf_layout  # noqa: E402


def main():
    insp = vi_b200.Inspector(0)
    p = vi_b200.default_params(threshold=8, min_area=0, erode_px=1)
    small = [((32 + 128 * i, 32 + 128 * j, 96, 96), j * 6 + i) for j in range(4) for i in range(6)]
    fr = np.stack([synth.make_frame(700 + i, [b for b, _ in small], H=576, W=832, inset=5, jitter=2, salt_p=s)
                   for i, s in enumerate((0.02, 0.15, 0.3))])
    insp.configure(Grid(boxes=small), is_reference=True)
    for k in (1, 8, 1024):
        tab = torch.empty((3 * len(small), k, 40), dtype=torch.uint8, device="cuda")
        insp.inspect_batch(torch.from_numpy(fr).cuda(), p, defect_blobs=tab)
    units = ARENA_UNITS + [(2048, 1500, 3)]
    boxes, _, bottom = shelf_layout(units, 2100)
    n = frames_for(len(units), torch.cuda.get_device_properties(0).multi_processor_count)
    fr = make_frames(boxes, n, bottom + 8, 2112, 1100)
    (x, y, w, h), _ = boxes[-1]
    inner = fr[0, y + 10:y + h - 10, x + 10:x + w - 10]
    inner[np.random.default_rng(5).random(inner.shape) < 0.25] = 255
    insp.configure(Grid(boxes=boxes), is_reference=True)
    tab = torch.empty((n * len(units), 1024, 40), dtype=torch.uint8, device="cuda")
    insp.inspect_batch(torch.from_numpy(fr).cuda(), p, defect_blobs=tab)
    torch.cuda.synchronize()
    word = C.c_uint32(12345)
    _lib.check(insp._lib.vi_debug_check_word(insp._ctx, C.byref(word)))
    print("check_word", int(word.value))


if __name__ == "__main__":
    main()
