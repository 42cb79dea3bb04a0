"""Runs the segmentation-only batch under the self-checked library (libvi_b200_checked.so) and prints the check word
(0 = no bound was violated): G1 on the segmentation kernel (tensor boxes) and with row copies on a strided view,
exclusions with the centroid shift on the general kernel, and the arena kernel with a 2048 x 1500 unit.  Started by
tests/test_gpu_segment_batch.py::test_checked_build_over_segment_batches with VI_B200_LIB=checked."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
assert os.environ.get("VI_B200_LIB") == "checked"

import torch  # noqa: E402
import vi_b200  # noqa: E402
from vi_b200 import _lib  # noqa: E402
from vi_b200.grid import Grid, ref_centroids_from_records  # noqa: E402
from test_gpu_unit_sequences import ARENA_UNITS, EXCL, G1, G2, frames_for, make_frames, shelf_layout  # noqa: E402


def main():
    insp = vi_b200.Inspector(0)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    for units, seed in ((G1, 3000), (G2, 3100)):
        boxes, _, bottom = shelf_layout(units, 1008)
        n = frames_for(len(units), sms)
        fr = make_frames(boxes, n, bottom + 8, 1024, seed)
        H = bottom + 8
        big = torch.zeros((n, H + 32, 1024 + 64), dtype=torch.uint8, device="cuda")
        big[:, :H, :1024] = torch.from_numpy(fr).cuda()
        insp.configure(Grid(boxes=boxes, exclusions=EXCL), is_reference=True)
        rec, _ = insp.segment_batch(big[:, :H, :1024])
        torch.cuda.synchronize()
        refc = ref_centroids_from_records(rec.cpu().numpy().view(vi_b200.RECORD_DTYPE))
        insp.configure(Grid(boxes=boxes, exclusions=EXCL, ref_centroids=refc), is_reference=False)
        insp.segment_batch(big[:, :H, :1024], vi_b200.default_params(gaussian_blur=5, morph_kernel=5))
        insp.segment_batch_host(fr, mask_format="packed")
    units = ARENA_UNITS + [(2048, 1500, 3)]
    boxes, _, bottom = shelf_layout(units, 2100)
    n = frames_for(len(units), sms)
    fr = make_frames(boxes, n, bottom + 8, 2112, 3200)
    insp.configure(Grid(boxes=boxes, exclusions=EXCL), is_reference=True)
    insp.segment_batch(torch.from_numpy(fr).cuda())
    torch.cuda.synchronize()
    word = C.c_uint32(12345)
    _lib.check(insp._lib.vi_debug_check_word(insp._ctx, C.byref(word)))
    print("check_word", int(word.value))


if __name__ == "__main__":
    main()
