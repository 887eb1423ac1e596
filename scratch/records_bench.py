"""Feature-point records against the full host results, and the records kernel's own device time.

  e2e      run_host_records against run_host on 64 x 1080p frames (scale sqrt2, 6 levels) from page-locked host memory,
           BGR and NV12, float32 and float16 outputs: all eight arms alternated in one process, medians and ranges,
           beside the concurrent pinned H2D + D2H copy probe of bench.py's e2e.link (taken after each round)
  kernel   point_records_kernel alone, after one run_frames(out=...) has left points, count and gray: CUDA events over
           back-to-back launches, and its duration from torch.profiler in a separate pass; at 64 x 1080p (3
           orientations) and 16 x 3840x2160 with a 16-orientation bank (8 levels), float32 and float16

The card's name and power limit are read in the same process. Writes one JSON file (--out).

    python scratch/records_bench.py --out records_bench.json [--runs 8] [--e2e-steps 5]
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
from half_bench import card, link_probe, summary   # noqa: E402
from pysilent_b200 import LineEndPipeline, _ops   # noqa: E402

SCALE = 2 ** .5
DTYPES = (("float32", torch.float32), ("float16", torch.float16))


def pinned_copy(a):
    t = torch.empty(a.shape, dtype=torch.uint8, pin_memory=True)
    t.numpy()[...] = a
    return t.numpy()


def e2e(bgr, nv12, runs, steps, dev):
    arms = {}
    for fmt, frames in (("bgr", bgr), ("nv12", nv12)):
        for dname, dt in DTYPES:
            pipe = LineEndPipeline(zoom_ratio=SCALE, out_dtype=dt, frame_format=fmt)
            full = pipe.run_host(frames)
            o = torch.empty(full.orient.shape, dtype=dt, pin_memory=True).numpy()
            e = torch.empty(full.orient.shape, dtype=dt, pin_memory=True).numpy()
            rec = pipe.run_host_records(frames)
            assert np.array_equal(rec.points, full.points), (fmt, dname)
            key = "%s_%s" % (fmt, dname)
            arms[key + "_run_host"] = ((lambda p, o, e, f: lambda: p.run_host(f, o, e))(pipe, o, e, frames),
                                       frames.nbytes, o.nbytes + e.nbytes)
            d2h = sum(a.nbytes for a in rec[:3]) + rec.gray.nbytes * (1 + 2 * rec.orient.shape[1])
            arms[key + "_run_host_records"] = ((lambda p, f: lambda: p.run_host_records(f))(pipe, frames),
                                               frames.nbytes, d2h)
            arms[key + "_run_host"][0]()
            arms[key + "_run_host_records"][0]()
    ms = {k: [] for k in arms}
    probes = []
    for _ in range(runs):
        for k, (fn, _, _) in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
            ms[k].append((time.perf_counter() - t0) * 1000.0 / steps)
        probes.append(link_probe(dev))
    probe = statistics.median(probes)
    b = bgr.shape[0]
    out = {}
    for k, (_, h2d, d2h) in arms.items():
        med = statistics.median(ms[k])
        out[k] = {"ms_per_call": summary(ms[k]), "frames_per_s": b / (med * 1e-3), "h2d_bytes": h2d, "d2h_bytes": d2h,
                  "larger_direction_gbs": max(h2d, d2h) / (med * 1e-3) / 1e9,
                  "frac_of_probe": max(h2d, d2h) / (med * 1e-3) / 1e9 / probe}
    for fmt in ("bgr", "nv12"):
        for dname, _ in DTYPES:
            key = "%s_%s" % (fmt, dname)
            out[key + "_speedup"] = (statistics.median(ms[key + "_run_host"]) /
                                     statistics.median(ms[key + "_run_host_records"]))
    out["link_probe_gbs_each_way"] = summary(probes)
    return out


def kernel_time(frames, launches, **pipe_kw):
    """point_records_kernel alone on the points, count and gray one run_frames call left in the plan."""
    res = {}
    for dname, dt in DTYPES:
        pipe = LineEndPipeline(zoom_ratio=SCALE, out_dtype=dt, **pipe_kw)
        full = pipe.run_frames(frames)
        plan = pipe.plan_for(frames)
        b, n = int(frames.shape[0]), int(full.orient.shape[0])
        cap = max(64 * n, 1024)
        bufs = (torch.empty_like(full.orient), torch.empty_like(full.padded_line_end),
                torch.empty((cap, 4), dtype=torch.int64, device=frames.device),
                torch.zeros(1, dtype=torch.int64, device=frames.device))
        rec = pipe.run_frames_records(frames)
        pipe.run_frames(frames, out=bufs)
        orient, line_end, points, count = bufs
        c = int(orient.shape[3])
        offs = torch.empty(b + 1, dtype=torch.int64, device=frames.device)
        yx = torch.empty((cap, 2), device=frames.device)
        vals = torch.empty((cap, 1 + 2 * c), device=frames.device)
        fn = lambda: _ops.point_records(plan, b, points, count, orient, line_end, None, offs, yx, vals)  # noqa: E731
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        per = []
        for _ in range(5):
            a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(launches):
                fn()
            z.record()
            torch.cuda.synchronize()
            per.append(a.elapsed_time(z) / launches)
        from torch.autograd import DeviceType
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(50):
                fn()
            torch.cuda.synchronize()
        durs = [e.time_range.elapsed_us() for e in prof.events()
                if e.device_type == DeviceType.CUDA and "point_records_kernel" in e.name]
        res[dname] = {"records": int(count.item()), "records_equal_run_frames_records": bool(
                          torch.equal(points[:len(rec.points)], rec.points)),
                      "events_ms_per_launch_back_to_back": summary(per),
                      "profiler_kernel_us": summary(durs) if durs else None, "kernels_profiled": len(durs)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=8)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=200)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "records_bench.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    record = {"card": card(), "runs": args.runs, "alternated": True}
    rs = np.random.RandomState(3000)
    bgr = pinned_copy(rs.randint(0, 256, size=(64, 1080, 1920, 3), dtype=np.uint8))
    nv12 = pinned_copy(rs.randint(0, 256, size=(64, 1620, 1920), dtype=np.uint8))
    record["kernel_c3"] = {"workload": "64 x 1080p uint8, scale sqrt2, 6 levels, 3 orientations",
                           **kernel_time(torch.from_numpy(bgr).to(dev), args.launches)}
    c4 = torch.from_numpy(rs.randint(0, 256, size=(16, 2160, 3840, 3), dtype=np.uint8)).to(dev)
    record["kernel_c4_bank16"] = {"workload": "16 x 3840x2160 uint8, scale sqrt2, 8 levels, 16 orientations",
                                  **kernel_time(c4, args.launches, orientations=16)}
    del c4
    torch.cuda.empty_cache()
    record["e2e"] = {"workload": "64 x 1080p from page-locked host memory (BGR uint8 [64,1080,1920,3] or NV12 "
                                 "[64,1620,1920]), scale sqrt2, 6 levels; run_host into page-locked outputs",
                     "steps_per_run": args.e2e_steps, **e2e(bgr, nv12, args.runs, args.e2e_steps, dev)}
    record["card_after"] = card()
    with open(args.out, "w") as f:
        json.dump(record, f, indent=1)
    for k in ("kernel_c3", "kernel_c4_bank16"):
        for dname, _ in DTYPES:
            r = record[k][dname]
            print("%s %s: %d records, %.4f ms/launch back to back, profiler %s us" % (
                k, dname, r["records"], r["events_ms_per_launch_back_to_back"]["median"],
                "%.2f" % r["profiler_kernel_us"]["median"] if r["profiler_kernel_us"] else "n/a"))
    e = record["e2e"]
    for fmt in ("bgr", "nv12"):
        for dname, _ in DTYPES:
            key = "%s_%s" % (fmt, dname)
            print("%s: run_host %.2f ms (%.3f of probe), records %.2f ms (%.3f of probe), x%.3f" % (
                key, e[key + "_run_host"]["ms_per_call"]["median"], e[key + "_run_host"]["frac_of_probe"],
                e[key + "_run_host_records"]["ms_per_call"]["median"], e[key + "_run_host_records"]["frac_of_probe"],
                e[key + "_speedup"]))
    print("probe GB/s each way: %.1f" % e["link_probe_gbs_each_way"]["median"])


if __name__ == "__main__":
    main()
