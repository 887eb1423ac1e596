"""Peak feature points: how many a batch yields, the peak emit's kernel times, and what peaks cost a pipeline step and
run_host_records, against the region emit.

  kernels  the five kernels of silent_plan_peak_points alone (level_threshold_kernel, peak_count_kernel,
           scan_level_kernel, peak_base_kernel, peak_write_kernel), after one run_frames(out=...) has left the plan's
           gray, from torch.profiler (median kernel duration over LAUNCHES launches, per run), at p = 0.1, 0.5 and 0.9 on
           64 x 1080p BGR uint8 frames with float32 outputs (3 orientations, 6 levels) and 16 x 3840x2160 with a
           16-orientation bank (8 levels); with the bytes of gray each kernel reads (the threshold reads each level once,
           the count and write passes read rows y - 1, y and y + 1, counted once) and the points found and written.
  step     run_frames(out=...) device time per step (CUDA events), peaks at p = 0.5 against the region emit, the two arms
           alternated in one process, on the 64 x 1080p frames.
  e2e      run_host_records(patch_radius=4) on the 64 x 1080p frames from page-locked host memory, with peaks at p = 0.1
           and 0.5 against without (region maxima), alternated, host clock around calls that synchronise. (At p = 0.9
           the 2.3 M points' 9 x 9 patches alone are 5.3 GB: a measurement of the download, not of the emit.)

The card's name and power limit are read in the same process. Writes one JSON file (--out).

    python scratch/peaks_bench.py --out peaks_bench.json [--runs 5] [--steps 10]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scratch"))
from half_bench import card, summary, time_device   # noqa: E402
from pysilent_b200 import LineEndPipeline, _ops   # noqa: E402

SCALE = 2 ** .5
PERCENTS = (0.1, 0.5, 0.9)
KERNELS = ("level_threshold_kernel", "peak_count_kernel", "scan_level_kernel", "peak_base_kernel", "peak_write_kernel")
LAUNCHES = 30


def profiled(fn):
    """Median torch.profiler duration (µs) of each of KERNELS over LAUNCHES calls of ``fn``."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(LAUNCHES):
            fn()
        torch.cuda.synchronize()
    out = {}
    for k in KERNELS:
        durs = [e.time_range.elapsed_us() for e in prof.events() if e.device_type == DeviceType.CUDA and k in e.name]
        assert len(durs) == LAUNCHES, (k, len(durs))
        out[k] = statistics.median(durs)
    return out


def kernel_time(frames, runs, **pipe_kw):
    pipe = LineEndPipeline(zoom_ratio=SCALE, peaks=0.5, **pipe_kw)
    full = pipe.run_frames(frames, want_points=False)
    plan = pipe.plan_for(frames)
    b, n = int(frames.shape[0]), int(full.orient.shape[0])
    dev = frames.device
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    pipe.run_frames(frames, out=(full.orient, full.padded_line_end, torch.empty((0, 4), dtype=torch.int64, device=dev),
                                 count))   # the plan's gray of these frames
    gray_bytes = n * plan.h * plan.w * 4
    res = {"levels": n, "level_hw": [plan.h, plan.w], "gray_bytes": gray_bytes}
    for p in PERCENTS:
        _ops.plan_peak_points(plan, b, p, torch.empty((0, 4), dtype=torch.int64, device=dev), count)
        total = int(count.item())
        points = torch.empty((total, 4), dtype=torch.int64, device=dev)
        fn = lambda: _ops.plan_peak_points(plan, b, p, points, count)  # noqa: E731
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        per = [profiled(fn) for _ in range(runs)]
        med = {k: statistics.median(r[k] for r in per) for k in KERNELS}
        emit_us = sum(med.values())
        res["p=%g" % p] = {
            "points": total, "points_per_level": total / n,
            "rows_with_points": int(torch.unique(points[:, 0] * plan.h + points[:, 1]).numel()),
            "points_bytes_written": total * 32,
            "profiler_kernel_us_median": med, "per_run": per,
            "sum_of_kernel_us": emit_us,
            "gray_read_gbs": {"level_threshold_kernel": gray_bytes / med["level_threshold_kernel"] / 1e3,
                              "peak_count_kernel": gray_bytes / med["peak_count_kernel"] / 1e3,
                              "peak_write_kernel": gray_bytes / med["peak_write_kernel"] / 1e3}}
    return res


def step_time(frames, runs, steps):
    dev = frames.device
    arms = {}
    for name, peaks in (("region", None), ("peaks_0.5", 0.5)):
        pipe = LineEndPipeline(zoom_ratio=SCALE, peaks=peaks)
        full = pipe.run_frames(frames, points_capacity=1 << 22)
        cap = max(len(full.points), 1024)
        out = (torch.empty_like(full.orient), torch.empty_like(full.padded_line_end),
               torch.empty((cap, 4), dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev))
        arms[name] = ((lambda pipe, out: lambda: pipe.run_frames(frames, out=out))(pipe, out), len(full.points))
    for fn, _ in arms.values():
        for _ in range(3):
            fn()
    ms = {k: [] for k in arms}
    for _ in range(runs):
        for k, (fn, _) in arms.items():
            ms[k].append(time_device(fn, steps))
    return {k: {"points": arms[k][1], "ms_per_step": summary(ms[k])} for k in arms}


def e2e(bgr, runs, steps):
    arms = {}
    for name, peaks in (("region", None), ("peaks_0.1", 0.1), ("peaks_0.5", 0.5)):
        pipe = LineEndPipeline(zoom_ratio=SCALE, peaks=peaks)
        rec = pipe.run_host_records(bgr, patch_radius=4)
        d2h = sum(a.nbytes for a in rec[:3]) + rec.gray.nbytes * (1 + 2 * rec.orient.shape[-1])
        arms[name] = ((lambda pipe: lambda: pipe.run_host_records(bgr, patch_radius=4))(pipe), len(rec.points), d2h)
    ms = {k: [] for k in arms}
    for _ in range(runs):
        for k, (fn, _, _) in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
            ms[k].append((time.perf_counter() - t0) * 1000.0 / steps)
    return {k: {"points": pts, "d2h_bytes": d2h, "h2d_bytes": bgr.nbytes, "ms_per_call": summary(ms[k])}
            for k, (_, pts, d2h) in arms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "peaks_bench.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    record = {"card": card(), "runs": args.runs, "launches_per_run": LAUNCHES}
    rs = np.random.RandomState(3000)   # the frames of records_bench.py
    host = torch.empty((64, 1080, 1920, 3), dtype=torch.uint8, pin_memory=True)
    host.numpy()[...] = rs.randint(0, 256, size=(64, 1080, 1920, 3), dtype=np.uint8)
    bgr = host.numpy()
    rs.randint(0, 256, size=(64, 1620, 1920), dtype=np.uint8)   # records_bench.py's NV12 draw: its 4K frames follow
    frames = host.to(dev)
    record["kernels_c3"] = {"workload": "64 x 1080p BGR uint8, scale sqrt2, 6 levels, 3 orientations, float32 outputs",
                            **kernel_time(frames, args.runs)}
    record["step"] = {"workload": "run_frames(out=...) on 64 x 1080p BGR uint8, float32 outputs, capacity = the points",
                      "steps_per_run": args.steps, **step_time(frames, args.runs, args.steps)}
    del frames
    c4 = torch.from_numpy(rs.randint(0, 256, size=(16, 2160, 3840, 3), dtype=np.uint8)).to(dev)
    record["kernels_c4_bank16"] = {"workload": "16 x 3840x2160 uint8, scale sqrt2, 8 levels, 16 orientations, float32 "
                                                "outputs", **kernel_time(c4, args.runs, orientations=16)}
    del c4
    torch.cuda.empty_cache()
    record["e2e"] = {"workload": "run_host_records(patch_radius=4) on 64 x 1080p BGR uint8 from page-locked host "
                                 "memory, float32", "steps_per_run": 3, **e2e(bgr, args.runs, 3)}
    record["card_after"] = card()
    with open(args.out, "w") as f:
        json.dump(record, f, indent=1)
    print(json.dumps(record["card"]))
    for k in ("kernels_c3", "kernels_c4_bank16"):
        for p in PERCENTS:
            r = record[k]["p=%g" % p]
            print("%s p=%g: %d points (%.1f per level), %s" % (
                k, p, r["points"], r["points_per_level"],
                ", ".join("%s %.2f" % (a.replace("_kernel", ""), v) for a, v in r["profiler_kernel_us_median"].items())))
    for k in ("step", "e2e"):
        for arm, v in record[k].items():
            if isinstance(v, dict):
                m = v.get("ms_per_step", v.get("ms_per_call"))
                print("%s %s: %d points, %.3f ms [%.3f-%.3f]" % (k, arm, v["points"], m["median"], m["min"], m["max"]))


if __name__ == "__main__":
    main()
