"""Cost of the kept-defect-component table (vi_set_defect_blob_output): each leg alternates the table off and on in
one process and prints the median of the per-round times of both.
    python tools/blob_bench.py [--rounds R]
  configs[1]: 64 frames of the grid.json grid (3,072 units of 316x315), device call, K = 64;
  config 5: one 16384x12000 frame of 11,811 salted 96x96 units, threshold 8 / min-area 0 / erode 1, K = 1024;
  host: configs[1]'s 64 frames (pinned) through inspect_batch_host, records only against records plus the table (K = 64)."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import vi_b200  # noqa: E402
from vi_b200 import synth  # noqa: E402
from vi_b200.grid import Grid, generate_grid  # noqa: E402


def device_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def alternate(name, units, off, on, rounds, reps, timer=device_ms):
    off(); on(); torch.cuda.synchronize()
    t_off, t_on = [], []
    for _ in range(rounds):
        t_off.append(timer(off, reps))
        t_on.append(timer(on, reps))
    a, b = float(np.median(t_off)), float(np.median(t_on))
    print(f"{name}: off {a:.3f} ms ({units / a * 1e3:,.0f} units/s, spread {min(t_off):.3f}-{max(t_off):.3f}), "
          f"on {b:.3f} ms ({units / b * 1e3:,.0f} units/s, spread {min(t_on):.3f}-{max(t_on):.3f}), cost {100 * (b / a - 1):+.2f} %")


def host_ms(fn, reps):
    import time
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    print(torch.cuda.get_device_name(0))
    boxes = generate_grid((251, 232, 316, 315), 4, 6, 2, 1, 133, 136, 252, 0)
    frames = np.stack([synth.make_frame(1000 + i, [b for b, _ in boxes]) for i in range(64)])
    insp = vi_b200.Inspector(0)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    p = vi_b200.default_params()
    d = torch.from_numpy(frames).cuda()
    n = 64 * insp.n_units
    rec = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    seg = torch.empty(64 * insp.unit_pixels, dtype=torch.uint8, device="cuda")
    dfm = torch.empty_like(seg)
    tab = torch.empty((n, 64, 40), dtype=torch.uint8, device="cuda")
    alternate("configs[1] device, K=64", n,
              lambda: insp.inspect_batch(d, p, seg, dfm, rec),
              lambda: insp.inspect_batch(d, p, seg, dfm, rec, defect_blobs=tab), args.rounds, 5)
    r = rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    print(f"  kept components per unit: mean {r['n_kept'].mean():.2f}, max {r['n_kept'].max()}")
    hf = torch.from_numpy(frames).pin_memory().numpy()             # pinned, as bench.py's e2e legs
    alternate("configs[1] host records-only, K=64", n,
              lambda: insp.inspect_batch_host(hf, p, mask_format="none"),
              lambda: insp.inspect_batch_host(hf, p, mask_format="none", max_blobs=64), args.rounds, 2, host_ms)
    del d, seg, dfm, tab, rec
    torch.cuda.empty_cache()

    b5 = synth.dense_grid_boxes()
    f5 = synth.make_frame(7, b5, H=12000, W=16384, inset=8, salt_p=0.02)
    i5 = vi_b200.Inspector(0)
    i5.configure(Grid(boxes=[(b, i) for i, b in enumerate(b5)]), is_reference=True)
    p5 = vi_b200.default_params(threshold=8, min_area=0, erode_px=1)
    d5 = torch.from_numpy(f5[None]).cuda()
    n5 = len(b5)
    rec5 = torch.empty((n5, 64), dtype=torch.uint8, device="cuda")
    seg5 = torch.empty(i5.unit_pixels, dtype=torch.uint8, device="cuda")
    dfm5 = torch.empty_like(seg5)
    tab5 = torch.empty((n5, 1024, 40), dtype=torch.uint8, device="cuda")
    alternate("config 5 device, K=1024", n5,
              lambda: i5.inspect_batch(d5, p5, seg5, dfm5, rec5),
              lambda: i5.inspect_batch(d5, p5, seg5, dfm5, rec5, defect_blobs=tab5), args.rounds, 5)
    r5 = rec5.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    print(f"  kept components per unit: mean {r5['n_kept'].mean():.2f}, max {r5['n_kept'].max()}")


if __name__ == "__main__":
    main()
