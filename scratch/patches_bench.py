"""Feature-point patches: the gather kernel's device time at several radii, and run_host_records with patches against
records and against the full host results.

  kernel   point_records_kernel alone, after one run_frames(out=...) has left points, count and gray, from
           torch.profiler (kernel durations, 50 launches per arm, arms alternated over --runs rounds): at 64 x 1080p (3
           orientations) and 16 x 3840x2160 with a 16-orientation bank (8 levels), float32 and float16. Arms:
             records       silent_point_records, capacity 64 rows per level (records_bench.py's launch)
             patches_r0    silent_point_patches at radius 0, the same capacity (the same launch through the new entry)
             exact_rR      silent_point_patches at radius R = 0, 2, 4, 8 with capacity = the points found (what
                           run_frames_records(patch_radius=R) launches without out=)
             records_into_r0_buffer, r0_into_records_buffer
                           the first two arms with their values buffers exchanged (placement against code)
             parent_records
                           with --parent-lib: silent_point_records of the parent commit's library, loaded beside this
                           one, on the same plan, points and buffers as the records arm (today's kernel, same process)
           The arms' order rotates by one each round.
  e2e      on 64 x 1080p BGR uint8 frames (scale sqrt2, 6 levels) from page-locked host memory, float32 and float16
           outputs: run_host_records(patch_radius=4), run_host_records() and run_host into page-locked outputs, all six
           arms alternated in one process, medians and ranges, with the bytes each call moves, beside the concurrent
           pinned H2D + D2H copy probe of bench.py's e2e.link (taken after each round)

The card's name and power limit are read in the same process. Writes one JSON file (--out).

    python scratch/patches_bench.py --out patches_bench.json [--runs 8] [--e2e-steps 5] [--parent-lib PATH]
"""
import argparse
import ctypes
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
from pysilent_b200 import LineEndPipeline, _lib, _ops   # noqa: E402

SCALE = 2 ** .5
DTYPES = (("float32", torch.float32), ("float16", torch.float16))
RADII = (0, 2, 4, 8)
LAUNCHES = 50
PARENT = None   # the parent commit's library (--parent-lib)


def parent_records(plan, b, points, count, orient, line_end, offs, yx, values):
    """silent_point_records of the parent's library on this library's plan (plan.h is the same in both)."""
    p = _ops.ptr
    half = int(orient.dtype == torch.float16)
    rc = PARENT.silent_point_records(plan.handle, b, p(points), p(count), int(points.shape[0]), p(orient), p(line_end),
                                     int(orient.shape[3]), half, None, p(offs), p(yx), p(values), _ops.stream_ptr())
    assert rc == 0, rc
    return offs, yx, values


def pinned_copy(a):
    t = torch.empty(a.shape, dtype=torch.uint8, pin_memory=True)
    t.numpy()[...] = a
    return t.numpy()


def profiled_us(fn, name):
    """Median torch.profiler duration (µs) of the kernels called ``name`` over LAUNCHES calls of ``fn``."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(LAUNCHES):
            fn()
        torch.cuda.synchronize()
    durs = [e.time_range.elapsed_us() for e in prof.events() if e.device_type == DeviceType.CUDA and name in e.name]
    assert len(durs) == LAUNCHES, (name, len(durs))
    return statistics.median(durs)


def kernel_time(frames, runs, **pipe_kw):
    res = {}
    for dname, dt in DTYPES:
        pipe = LineEndPipeline(zoom_ratio=SCALE, out_dtype=dt, **pipe_kw)
        full = pipe.run_frames(frames)
        plan = pipe.plan_for(frames)
        b, n = int(frames.shape[0]), int(full.orient.shape[0])
        dev = frames.device
        cap = max(64 * n, 1024)
        bufs = (torch.empty_like(full.orient), torch.empty_like(full.padded_line_end),
                torch.empty((cap, 4), dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev))
        pipe.run_frames(frames, out=bufs)
        orient, line_end, points, count = bufs
        total = int(count.item())
        c = int(orient.shape[3])
        offs = torch.empty(b + 1, dtype=torch.int64, device=dev)
        yx = torch.empty((cap, 2), device=dev)
        v_rec, v_r0 = torch.empty((cap, 1 + 2 * c), device=dev), torch.empty((cap, 1, 1, 1 + 2 * c), device=dev)
        rec = lambda v: lambda: _ops.point_records(plan, b, points, count, orient, line_end, None, offs, yx, v)  # noqa
        r0 = lambda v: lambda: _ops.point_records(plan, b, points, count, orient, line_end, None, offs, yx, v,  # noqa
                                                  radius=0)
        arms = {"records": rec(v_rec), "patches_r0": r0(v_r0), "records_into_r0_buffer": rec(v_r0.view(v_rec.shape)),
                "r0_into_records_buffer": r0(v_rec.view(v_r0.shape))}
        if PARENT is not None:
            arms["parent_records"] = (lambda v: lambda: parent_records(plan, b, points, count, orient, line_end, offs,
                                                                       yx, v))(torch.empty_like(v_rec))
        exact = points[:total]
        for r in RADII:
            p = 2 * r + 1
            arms["exact_r%d" % r] = (lambda v, r: lambda: _ops.point_records(plan, b, exact, count, orient, line_end,
                                                                             None, offs, yx[:total], v, radius=r))(
                torch.empty((total, p, p, 1 + 2 * c), device=dev), r)
        # every arm's values at the points (the patch centres) against the records'
        want = arms["records"]()[2].clone()
        checks = {}
        for k, fn in arms.items():
            v = fn()[2]
            centre = v if v.dim() == 2 else v[:, v.shape[1] // 2, v.shape[2] // 2]
            checks[k] = bool(torch.equal(torch.nan_to_num(centre[:total], 7.0), torch.nan_to_num(want[:total], 7.0)))
        for fn in arms.values():
            for _ in range(10):
                fn()
        torch.cuda.synchronize()
        per = {k: [] for k in arms}
        names = list(arms)
        for i in range(runs):
            for k in names[i % len(names):] + names[:i % len(names)]:
                per[k].append(profiled_us(arms[k], "point_records_kernel"))
        res[dname] = {"records": total, "capacity_64_per_level": cap, "centre_equals_records": checks,
                      "values_bytes_written": {"exact_r%d" % r: total * (2 * r + 1) ** 2 * (1 + 2 * c) * 4
                                               for r in RADII},
                      "profiler_kernel_us_median_of_%d_per_run" % LAUNCHES: {k: summary(v) for k, v in per.items()}}
    return res


def e2e(bgr, runs, steps, dev):
    arms = {}
    for dname, dt in DTYPES:
        pipe = LineEndPipeline(zoom_ratio=SCALE, out_dtype=dt)
        full = pipe.run_host(bgr)
        o = torch.empty(full.orient.shape, dtype=dt, pin_memory=True).numpy()
        e = torch.empty(full.orient.shape, dtype=dt, pin_memory=True).numpy()
        rec = pipe.run_host_records(bgr)
        pat = pipe.run_host_records(bgr, patch_radius=4)
        assert np.array_equal(rec.points, full.points) and np.array_equal(pat.points, full.points), dname
        assert np.array_equal(pat.orient[:, 4, 4], rec.orient, equal_nan=True), dname
        nbytes = lambda r: sum(a.nbytes for a in r[:3]) + r.gray.nbytes * (1 + 2 * r.orient.shape[-1])  # noqa: E731
        arms[dname + "_run_host"] = ((lambda p, o, e: lambda: p.run_host(bgr, o, e))(pipe, o, e),
                                     o.nbytes + e.nbytes + full.points.nbytes)
        arms[dname + "_run_host_records"] = ((lambda p: lambda: p.run_host_records(bgr))(pipe), nbytes(rec))
        arms[dname + "_run_host_records_r4"] = ((lambda p: lambda: p.run_host_records(bgr, patch_radius=4))(pipe),
                                                nbytes(pat))
    for fn, _ in arms.values():
        fn()
    ms = {k: [] for k in arms}
    probes = []
    for _ in range(runs):
        for k, (fn, _) in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
            ms[k].append((time.perf_counter() - t0) * 1000.0 / steps)
        probes.append(link_probe(dev))
    b = bgr.shape[0]
    out = {k: {"ms_per_call": summary(ms[k]), "frames_per_s": b / (statistics.median(ms[k]) * 1e-3),
               "h2d_bytes": bgr.nbytes, "d2h_bytes": d2h} for k, (_, d2h) in arms.items()}
    out["link_probe_gbs_each_way"] = summary(probes)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=8)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--parent-lib", help="libsilent_b200.so of the parent commit, for the parent_records arm")
    args = ap.parse_args()
    global PARENT
    if args.parent_lib:
        PARENT = ctypes.CDLL(os.path.abspath(args.parent_lib))   # RTLD_LOCAL: its symbols stay apart from this one's
        PARENT.silent_point_records.restype = ctypes.c_int
        PARENT.silent_point_records.argtypes = _lib.lib().silent_point_records.argtypes
    assert torch.cuda.is_available(), "patches_bench.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    record = {"card": card(), "runs": args.runs, "alternated": True, "parent_lib": args.parent_lib}
    rs = np.random.RandomState(3000)   # the frames of records_bench.py
    bgr = pinned_copy(rs.randint(0, 256, size=(64, 1080, 1920, 3), dtype=np.uint8))
    rs.randint(0, 256, size=(64, 1620, 1920), dtype=np.uint8)   # records_bench.py's NV12 draw: its 4K frames follow
    record["kernel_c3"] = {"workload": "64 x 1080p uint8, scale sqrt2, 6 levels, 3 orientations",
                           **kernel_time(torch.from_numpy(bgr).to(dev), args.runs)}
    c4 = torch.from_numpy(rs.randint(0, 256, size=(16, 2160, 3840, 3), dtype=np.uint8)).to(dev)
    record["kernel_c4_bank16"] = {"workload": "16 x 3840x2160 uint8, scale sqrt2, 8 levels, 16 orientations",
                                  **kernel_time(c4, args.runs, orientations=16)}
    del c4
    torch.cuda.empty_cache()
    record["e2e"] = {"workload": "64 x 1080p BGR uint8 [64,1080,1920,3] from page-locked host memory, scale sqrt2, 6 "
                                 "levels; run_host into page-locked outputs", "steps_per_run": args.e2e_steps,
                     **e2e(bgr, args.runs, args.e2e_steps, dev)}
    record["card_after"] = card()
    with open(args.out, "w") as f:
        json.dump(record, f, indent=1)
    key = "profiler_kernel_us_median_of_%d_per_run" % LAUNCHES
    for k in ("kernel_c3", "kernel_c4_bank16"):
        for dname, _ in DTYPES:
            r = record[k][dname]
            print("%s %s: %d points, centre checks %s" % (k, dname, r["records"], all(r["centre_equals_records"].values())))
            print("   " + ", ".join("%s %.2f [%.2f-%.2f]" % (a, s["median"], s["min"], s["max"]) for a, s in r[key].items()))
    e = record["e2e"]
    for k, v in e.items():
        if isinstance(v, dict) and "d2h_bytes" in v:
            print("%s: %.2f ms [%.2f-%.2f], %d B down" % (k, v["ms_per_call"]["median"], v["ms_per_call"]["min"],
                                                       v["ms_per_call"]["max"], v["d2h_bytes"]))
    print("probe GB/s each way: %.1f" % e["link_probe_gbs_each_way"]["median"])


if __name__ == "__main__":
    main()
