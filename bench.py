#!/usr/bin/env python
"""bench.py -- the hot-path benchmark (BASELINE.json metric: units/s on synthetic
4096x3000 mold images with the reference's grid.json grid).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the full per-unit inspection path (segmentation +
defect pass + verdict) over one batch of `--images` (default 64 = configs[1])
synthetic frames per GPU.  `value` is measured with the frames already resident
in HBM; `e2e` goes through the host-buffer C-ABI call (pinned host frames in,
masks + records out, copies inside the timed region).  Multi-GPU (torchrun, one
process per GPU): configs[2], 1024 frames sharded by image; the per-unit record
table is gathered by the kernel itself over NVLink peer memory and verified on
rank 0 against an NCCL all-gather and a 1-rank run.

`--dump-outputs DIR` writes what the last timed step computed (see `dump_outputs`) as DIR/<name>.npy, so that two
builds of the project can be compared output for output on the same inputs.

`--impl reference` times the reference's own CPU path (the cv2 oracle port,
oracle/ref_cv2.py -- the reference itself needs PyQt6 and is absent on the GPU
box) on all host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# NCCL prints its version banner to stdout at NCCL_DEBUG=VERSION (set on the GPU boxes) and at WARN: stdout carries
# the JSON line only, so that level is dropped before torch / NCCL are loaded (INFO and above are left alone).
if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
    del os.environ["NCCL_DEBUG"]

import numpy as np

GRID_BASE = (251, 232, 316, 315)          # the reference's grid.json: 2 blocks x (4 x 6) units of 316x315
GRID_ARGS = (4, 6, 2, 1, 133, 136, 252, 0)
W, H = 4096, 3000
UNIT_PX = 316 * 315
ALGO_BYTES_PER_PX = 3                      # 1 B gray in + 1 B seg mask out + 1 B defect mask out (SURVEY 8d)


def grid_boxes():
    from vi_b200.grid import generate_grid
    return generate_grid(GRID_BASE, *GRID_ARGS)


# --------------------------------------------------------------------------- CPU arm
_CPU_FRAMES = None


def _cpu_init():
    import cv2
    cv2.setNumThreads(1)


def _cpu_one(i):
    from oracle import ref_cv2 as R
    recs, _, _ = R.inspect_frame(_CPU_FRAMES[i], grid_boxes(), R.Params(), (), None, True)
    return sum(1 for r in recs if r['status'] == R.STATUS_NG)


def cpu_reference_run(frames, cores, passes=1):
    """Units/s of the reference CPU path on `cores` processes (images sharded); `passes` repeats the frame list."""
    import multiprocessing as mp
    global _CPU_FRAMES
    _CPU_FRAMES = frames
    n_units = len(grid_boxes())
    if cores <= 1:
        _cpu_init()
        t0 = time.perf_counter()
        ng = [_cpu_one(i) for _ in range(passes) for i in range(len(frames))]
        dt = time.perf_counter() - t0
    else:
        ctx = mp.get_context('fork')
        with ctx.Pool(cores, initializer=_cpu_init) as pool:
            pool.map(_cpu_one, range(min(cores, len(frames))))      # warm the workers (imports, page-in)
            t0 = time.perf_counter()
            ng = pool.map(_cpu_one, [i for _ in range(passes) for i in range(len(frames))], chunksize=1)
            dt = time.perf_counter() - t0
    return passes * len(frames) * n_units / dt, dt, int(sum(ng))


def make_frames(seeds):
    from vi_b200 import synth
    boxes = [b for b, _ in grid_boxes()]
    return [synth.make_frame(s, boxes, H=H, W=W) for s in seeds]


# --------------------------------------------------------------------------- output dump
DUMP_MASK_UNITS = 48                       # units whose masks are dumped: both full mask sets are 612 MB at configs[1]
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, insp, rec, d_seg, d_def):
    """Writes the outputs of one batch call as float arrays: every record field as record_<field>.npy [images, units]
    (float64: the int32 fields and the float64 centroids are exact), and the seg / defect masks (0 or 255) of a fixed,
    seeded sample of the batch's units as seg_masks.npy / defect_masks.npy [k, h, w] float32, with the sampled
    (image, unit) pairs in sample_units.npy [k, 2]."""
    n_units = insp.n_units
    rec = rec.reshape(-1, n_units)
    arrays = {f"record_{k}": rec[k].astype(np.float64) for k in rec.dtype.names}
    n_all = rec.size
    pick = np.sort(np.random.default_rng(0).choice(n_all, size=min(DUMP_MASK_UNITS, n_all), replace=False))
    arrays["sample_units"] = np.stack([pick // n_units, pick % n_units], axis=1).astype(np.float64)
    for name, flat in (("seg_masks", d_seg), ("defect_masks", d_def)):
        arrays[name] = np.stack([insp.split_masks(flat, int(p // n_units))[int(p % n_units)].cpu().numpy()
                                 for p in pick]).astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"output dump of {total} bytes exceeds {DUMP_MAX_BYTES}"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for t, ln in self.lines:
            if t < t0 or t > t1 + 0.2:
                continue
            f = [x.strip() for x in ln.split(',')]
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "samples": len(sm),
                "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- frame ingest (streaming kernels)
def ingest_bench(insp, dev, n_img, peak, reps=10):
    """The two frame-ingest kernels (SURVEY n3) on n_img 4096x3000 frames: pure HBM streaming, reported against the
    same measured copy bandwidth as the main kernel (algorithmic bytes: 4+1 and 2+1 per pixel)."""
    import torch
    out = {}
    dst = torch.empty((n_img, H, W), dtype=torch.uint8, device=dev)
    for name, shape, dtype, bpp, fn in (("argb32", (n_img, H, W, 4), torch.uint8, 5, insp.ingest_argb32),
                                        ("gray16", (n_img, H, W), torch.int16, 3, insp.ingest_gray16)):
        src = torch.empty(shape, dtype=dtype, device=dev)
        src.view(torch.uint8).random_(0, 256)
        for _ in range(3):
            fn(src, out=dst)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn(src, out=dst)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        gbs = bpp * n_img * H * W / (ms * 1e-3) / 1e9
        out[name] = {"ms_per_launch": ms, "frame_gpix_per_s": n_img * H * W / (ms * 1e-3) / 1e9, "achieved": gbs, "peak": peak,
                     "unit": "GB/s", "frac": gbs / peak, "algorithmic_bytes_per_px": bpp, "frames": n_img}
        del src
    return out


# --------------------------------------------------------------------------- main arms
def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_frames = max(cores, 8) if args.ref_frames <= 0 else args.ref_frames
    n_frames = min(n_frames, 2 * cores)
    frames = make_frames(range(n_frames))
    vals = []
    for _ in range(args.warmup):
        cpu_reference_run(frames[:min(len(frames), cores)], cores)
    t_all = 0.0
    for _ in range(args.steps):
        v, dt, ng = cpu_reference_run(frames, cores, args.ref_passes)
        vals.append(v); t_all += dt
    value = float(np.mean(vals))
    sample = (f"{n_frames} frames x 48 units x {args.ref_passes} passes per step ({n_frames * 48 * args.ref_passes} units), "
              f"{cores} processes x 1 cv2 thread, oracle/ref_cv2.py (cv2 port of the reference path; the reference's per-unit Qt "
              f"conversions are omitted -- PyQt6 is absent -- which flatters the reference slightly)")
    out = {
        "impl": "reference", "metric": "units/s", "value": value, "unit": "units/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "configs[1]: 4096x3000 frames, grid.json grid (48 units of 316x315), defaults "
                               "(otsu, blur 3, morph 3, thr 24, min-area 20, erode 6); bounded sample", "images_per_step": n_frames},
        "gpix_per_s": value * UNIT_PX / 1e9,
        "cpu_baseline": {"value": value, "unit": "units/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "units/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def run_gpu_arm(args, rank, world, local_rank):
    from vi_b200 import numa
    binding = numa.bind_to_gpu(local_rank) if not args.no_bind else {"bound": False, "source": "off"}   # before any pinned allocation
    import torch
    import vi_b200
    from vi_b200 import dist as vdist
    from vi_b200.grid import Grid
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    boxes = grid_boxes()
    n_units = len(boxes)
    insp = vi_b200.Inspector(local_rank)
    insp.configure(Grid(boxes=boxes), is_reference=True)
    params = vi_b200.default_params()

    # Workload.  N = 1: configs[1], one batch of --images frames.  N > 1: configs[2], --global-images frames sharded by
    # image (global image i -> rank i % world, vi_b200.dist.shard_images); every rank holds its slice.  Global image i
    # shows synthetic frame seed i % --distinct, so that rank 0 can check the gathered table against a 1-rank run.
    n_dist = min(args.distinct, args.images if world == 1 else args.global_images)
    uniq = make_frames(range(n_dist))
    if world == 1:
        n_global = args.images
        mine = list(range(n_global))
    else:
        n_global = args.global_images
        mine = vdist.shard_images(n_global, rank, world)
    n_img = len(mine)
    h_frames_t = torch.empty((n_img, H, W), dtype=torch.uint8, pin_memory=True)
    h_frames = h_frames_t.numpy()
    for k, gi in enumerate(mine):
        h_frames[k] = uniq[gi % n_dist]
    d_frames = h_frames_t.to(dev, non_blocking=True)
    total_px = n_img * insp.unit_pixels
    d_seg = torch.empty(total_px, dtype=torch.uint8, device=dev)
    d_def = torch.empty(total_px, dtype=torch.uint8, device=dev)
    d_rec = torch.empty((n_img * n_units, 64), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    # Multi-GPU: the record table is gathered by the kernel itself -- every record is also stored into every rank's
    # peer-mapped table over NVLink (vi_b200.dist.RecordExchange); no collective runs inside a step.
    exch = vdist.RecordExchange(insp, n_global) if world > 1 else None

    def step():
        insp.inspect_batch(d_frames, params, seg_masks=d_seg, defect_masks=d_def, records=d_rec)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    t1 = time.perf_counter()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop(t0, t1) if sampler else None
    ms_per_step = ms / args.steps
    units_per_step = n_global * n_units
    value = units_per_step / (ms_per_step * 1e-3)

    rec = d_rec.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(-1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, insp, rec, d_seg, d_def)
    ng_gpu = int((rec['status'] == vi_b200.STATUS_NG).sum())
    table_check = None
    if world > 1:
        # the kernel-gathered table == an NCCL all-gather of the ranks' record blocks == a 1-rank run of the same images
        exch.complete()
        table = exch.table()
        table_nccl = vdist.gather_record_table(d_rec, n_global, n_units)
        if rank == 0:
            insp1 = vi_b200.Inspector(local_rank)                     # no peers: plain single-GPU context
            insp1.configure(Grid(boxes=boxes), is_reference=True)
            d_u = torch.from_numpy(np.stack(uniq)).to(dev)
            r1, _, _ = insp1.inspect_batch(d_u, params)
            torch.cuda.synchronize()
            r1 = r1.cpu().numpy().view(vi_b200.RECORD_DTYPE).reshape(n_dist, n_units)
            table_1 = r1[np.arange(n_global) % n_dist].copy()
            table_1['image'] = np.arange(n_global)[:, None]
            for name, other in (("nccl all-gather", table_nccl), ("1-rank run", table_1)):
                for k in vi_b200.RECORD_DTYPE.names:
                    a_, b_ = table[k], other[k]
                    same = np.array_equal(a_, b_) or (a_.dtype.kind == 'f' and np.array_equal(np.isnan(a_), np.isnan(b_))
                                                      and np.array_equal(a_[~np.isnan(a_)], b_[~np.isnan(b_)]))
                    assert same, f"record table gathered by the kernel differs from the {name} in field {k}"
            ng_gpu = int((table['status'] == vi_b200.STATUS_NG).sum())
            table_check = (f"kernel-gathered table [{n_global} x {n_units}] equals the NCCL all-gather and the 1-rank run in every "
                           f"field ({ng_gpu} NG units)")
            del insp1, d_u

    # ---- e2e: host buffers through the C ABI, copies inside the timed region ----
    def e2e_leg(fmt, steps):
        per_img = {"bytes": insp.unit_pixels, "packed": insp.packed_bytes, "none": 0}[fmt]
        h_seg = torch.empty(max(1, n_img * per_img), dtype=torch.uint8, pin_memory=True).numpy()
        h_def = torch.empty(max(1, n_img * per_img), dtype=torch.uint8, pin_memory=True).numpy()
        h_rec = torch.empty(n_img * n_units * 64, dtype=torch.uint8, pin_memory=True).numpy().view(vi_b200.RECORD_DTYPE)
        gathered = [torch.empty_like(d_rec) for _ in range(world)] if world > 1 else None

        def once():
            insp.inspect_batch_host(h_frames, params, out=(h_rec, h_seg, h_def), mask_format=fmt)
            if world > 1:
                dist.all_gather(gathered, torch.from_numpy(h_rec.view(np.uint8).reshape(-1, 64)).to(dev))
        for _ in range(2):
            once()
        barrier()
        t0e = time.perf_counter()
        for _ in range(steps):
            once()
        barrier()
        s_ = (time.perf_counter() - t0e) / steps
        if world > 1:
            t_ = torch.tensor([s_], device=dev)
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            s_ = float(t_.item())
        assert np.array_equal(h_rec['status'], rec['status']), "host-buffer path and device-resident path disagree"
        mapped = os.environ.get("VI_HOST_UPLOAD", "") == "mapped"
        h2d = int(insp._lib.vi_host_upload_bytes(insp._ctx, n_img, 0 if mapped else W))
        return {"value": units_per_step / s_, "unit": "units/s", "ms_per_step": s_ * 1e3, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": int(2 * n_img * per_img + n_img * n_units * 64), "mask_format": fmt,
                "upload": "crop gather from mapped pinned frames" if mapped else "staged: frame rows covered by units"}

    if exch is not None:
        insp._lib.vi_set_record_peers(insp._ctx, None, 0, 1, 0)       # the host-buffer legs exchange records through NCCL
    e2e_steps = max(1, min(args.steps, 20 if world == 1 else 4))
    e2e = e2e_leg("bytes", e2e_steps)
    e2e_packed = e2e_leg("packed", e2e_steps) if not args.no_extra else None
    e2e_records = e2e_leg("none", e2e_steps) if not args.no_extra else None

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)"
        else:
            peak = 6650.0; peak_src = "fallback 6650 GB/s (of fallback)"
        ingest = None
        if world == 1 and not args.no_ingest:
            del d_seg, d_def
            torch.cuda.empty_cache()
            ingest = ingest_bench(insp, dev, min(n_img, 64), peak)
        algo_bytes_per_launch = ALGO_BYTES_PER_PX * n_img * insp.unit_pixels
        achieved = algo_bytes_per_launch / (ms_per_step * 1e-3) / 1e9      # per GPU: one launch per step per rank
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic = tj.get("dram_bytes_per_unit", 0) * n_img * n_units or tj.get("dram_bytes_per_launch")
        # CPU baseline: bounded sample on rank 0's host cores (N=1 only)
        cpu = None
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            n_s = min(max(cores, 4), n_dist, 2 * cores)
            v, dt, ng_cpu = cpu_reference_run(uniq[:n_s], cores, args.cpu_passes)
            ng_gpu_s = int((rec['status'][:n_s * n_units] == vi_b200.STATUS_NG).sum())
            assert ng_cpu == ng_gpu_s * args.cpu_passes, f"NG count differs: cpu {ng_cpu} vs gpu {ng_gpu_s} x {args.cpu_passes}"
            v1, dt1, _ = cpu_reference_run(uniq[:2], 1, 1)          # the reference as it really runs: one Python loop, one process
            cpu = {"value": v, "unit": "units/s", "cores": cores, "kind": "port", "single_process_units_per_s": v1,
                   "sample": f"{n_s} of the same frames x 48 units x {args.cpu_passes} passes ({n_s * n_units * args.cpu_passes} "
                             f"units, {dt:.1f} s), {cores} processes x 1 cv2 thread, oracle/ref_cv2.py (the reference's per-unit "
                             f"Qt conversions -- QPixmap.toImage, convertToFormat, QPixmap.fromImage -- are omitted: PyQt6 is "
                             f"absent, so this flatters the reference slightly); NG count per pass equals the GPU's ({ng_gpu_s})"}
        if world == 1:
            workload = ("configs[1]: batch of %d synthetic 4096x3000 frames, grid.json grid (48 units of 316x315), defaults "
                        "(otsu, blur 3, morph 3, thr 24, min-area 20, erode 6)" % n_img)
        else:
            workload = ("configs[2]: %d synthetic 4096x3000 frames sharded by image (i mod %d) across %d GPUs = %d per GPU, "
                        "grid.json grid (48 units of 316x315), defaults; record table gathered by the kernel over NVLink peer "
                        "memory, verified against an NCCL all-gather and a 1-rank run" % (n_global, world, world, n_img))
        out = {
            "metric": "units/s", "value": value, "unit": "units/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak" if world == 1 else "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload, "images_per_gpu": n_img, "global_images": n_global, "units_per_step": units_per_step,
                       "distinct_frames": n_dist,
                       "l2": "inputs (%.0f MB per step per GPU) exceed the 126 MB L2" % (n_img * H * W / 1e6),
                       "scaling_note": "N=1 is configs[1] (64 frames); N=2/4/8 split the same 1024-frame job (strong scaling); "
                                       "units/s is the whole job's either way",
                       "collective": ("none inside a step: records are stored into every rank's table by the kernel (peer memory); "
                                      "NCCL carries barriers, the timing all-reduce and the verification all-gather") if world > 1 else "none",
                       "host_binding": binding},
            "gpix_per_s": value * UNIT_PX / 1e9,
            "frame_gpix_per_s": value / n_units * W * H / 1e9,
            "ng_units": ng_gpu,
            "table_check": table_check,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": algo_bytes_per_launch, "kernel": "vi_unit_kernel"},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "e2e_packed_masks": e2e_packed,
            "e2e_records_only": e2e_records,
            "gpu_launches": args.steps,
            "ingest": ingest,
            "clocks": clocks,
        }
        print(json.dumps(out), flush=True)
    if exch is not None:
        exch.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--images", type=int, default=64, help="frames per step at N=1 (configs[1] = 64)")
    ap.add_argument("--global-images", type=int, default=1024, help="frames of the whole job at N>1 (configs[2] = 1024)")
    ap.add_argument("--no-bind", action="store_true", help="do not bind the process to the cores next to its GPU")
    ap.add_argument("--no-extra", action="store_true", help="skip the packed-mask and records-only e2e legs")
    ap.add_argument("--distinct", type=int, default=16, help="distinct synthetic frames (global image i shows frame i %% distinct)")
    ap.add_argument("--ref-frames", type=int, default=0, help="frames per step of the reference arm (0 = host cores)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-ingest", action="store_true", help="skip the frame-ingest streaming kernels")
    ap.add_argument("--cpu-passes", type=int, default=40, help="passes over the sample frames in the cpu_baseline leg (~10 s)")
    ap.add_argument("--ref-passes", type=int, default=8, help="passes over the sample frames per step of the reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's records and a seeded sample of its masks as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm keeps only NG counts")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    run_gpu_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
