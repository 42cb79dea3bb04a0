"""What the segmentation-only call saves: each leg alternates the full inspection and the segmentation-only call in one
process and prints the median (and spread) of the per-round times of both.
    python tools/seg_bench.py [--rounds R]
  configs[1] device: 64 frames of the grid.json grid (3,072 units of 316x315; the frames' bytes are printed: more than
    the 126 MB of L2), inspect_batch against segment_batch;
  configs[1] host: the same frames (pinned) through inspect_batch_host against segment_batch_host, in the bytes and the
    records-only formats.
Then the per-phase cycles of the segmentation kernel (its profiling instantiation)."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import vi_b200  # noqa: E402
from vi_b200 import _lib, synth  # noqa: E402
from vi_b200.grid import Grid, generate_grid  # noqa: E402

# phase slots of the segmentation path (vi_unit.cuh: pt.tick); slot 3 is the median stage's cell pass, empty here
SEG_PHASES = ["gather", "blur+hist", "otsu: estimate + exact scan", "(cell pass)", "threshold", "close/open",
              "hole fill", "centroid ccl", "excl+seg out"]


def device_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def host_ms(fn, reps):
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t) * 1e3 / reps


def alternate(name, units, full, seg, rounds, reps, timer=device_ms):
    full(); seg(); torch.cuda.synchronize()
    tf, ts = [], []
    for _ in range(rounds):
        tf.append(timer(full, reps))
        ts.append(timer(seg, reps))
    a, b = float(np.median(tf)), float(np.median(ts))
    print(f"{name}: inspect {a:.3f} ms ({units / a * 1e3:,.0f} units/s, spread {min(tf):.3f}-{max(tf):.3f}), "
          f"segment {b:.3f} ms ({units / b * 1e3:,.0f} units/s, spread {min(ts):.3f}-{max(ts):.3f}), "
          f"segment/inspect {b / a:.3f}")


def gpu_info():
    print("device:", torch.cuda.get_device_name(0))
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        print("nvidia-smi:", " | ".join(out.splitlines()))
    except Exception as e:                                             # noqa: BLE001
        print("nvidia-smi: not read:", e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    gpu_info()
    boxes = generate_grid((251, 232, 316, 315), 4, 6, 2, 1, 133, 136, 252, 0)
    frames = np.stack([synth.make_frame(1000 + i, [b for b, _ in boxes]) for i in range(64)])
    insp = vi_b200.Inspector(0)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    p = vi_b200.default_params()
    d = torch.from_numpy(frames).cuda()
    print(f"configs[1]: {frames.shape[0]} frames of {frames.shape[2]}x{frames.shape[1]}, {frames.nbytes / 1e6:.0f} MB")
    n = 64 * insp.n_units
    rec = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    seg = torch.empty(64 * insp.unit_pixels, dtype=torch.uint8, device="cuda")
    dfm = torch.empty_like(seg)
    alternate("configs[1] device", n, lambda: insp.inspect_batch(d, p, seg, dfm, rec),
              lambda: insp.segment_batch(d, p, seg, rec), args.rounds, 5)
    hf = torch.from_numpy(frames).pin_memory().numpy()             # pinned, as bench.py's e2e legs
    for fmt in ("bytes", "none"):
        alternate(f"configs[1] host, {fmt}", n, lambda: insp.inspect_batch_host(hf, p, mask_format=fmt),
                  lambda: insp.segment_batch_host(hf, p, mask_format=fmt), args.rounds, 2, host_ms)

    # per-phase cycles of the segmentation kernel (profiling instantiation: timers cost a little)
    prof = torch.zeros((n, 48), dtype=torch.int64, device="cuda")
    _lib.check(insp._lib.vi_debug_set_profile(insp._ctx, prof.data_ptr()))
    try:
        insp.segment_batch(d, p, seg, rec)
        torch.cuda.synchronize()
    finally:
        _lib.check(insp._lib.vi_debug_set_profile(insp._ctx, None))
    pr = prof.cpu().numpy().astype(np.float64)
    mean = pr.mean(0)
    print(f"segmentation kernel, mean cycles/unit over {n} units: {mean[:len(SEG_PHASES)].sum():.0f}")
    for i, nm in enumerate(SEG_PHASES):
        print(f"  {i:2d} {nm:30s} {mean[i]:10.0f}")
    print(f"  of which the exact Otsu scan (sub-phase slots 38-42): {pr[:, 38:43].sum(1).mean():.0f}")


if __name__ == "__main__":
    main()
