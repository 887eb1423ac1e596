"""float32 against float16 outputs (LineEndPipeline(out_dtype=...)), alternated in one process, on three workloads:

  c3      device step (ms) of run_frames with points: 64 x 1080p uint8 frames, scale sqrt2, 6 levels (BASELINE C3)
  c4      device step (ms) of run_frames on C4's frames (16 x 3840x2160, scale sqrt2, 8 levels) at bank widths 4, 8, 12, 16
  e2e     run_host on the 64 x 1080p frames from page-locked host buffers (frames/s), beside the concurrent pinned
          H2D + D2H copy probe of bench.py's e2e.link, and the larger direction's rate as a fraction of that probe

Each measurement is repeated --runs times per dtype, the two dtypes alternating; medians and ranges are reported. The
card's name and power limit are read in the same process. Writes one JSON file (--out).

    python scratch/half_bench.py --out half_bench.json [--runs 8] [--steps 20]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pysilent_b200 import LineEndPipeline   # noqa: E402

SCALE = 2 ** .5
DTYPES = (("float32", torch.float32), ("float16", torch.float16))


def card():
    q = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                text=True).splitlines()[torch.cuda.current_device()]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def summary(values):
    return {"median": statistics.median(values), "min": min(values), "max": max(values), "runs": values}


def time_device(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def device_steps(frames, runs, steps, **pipe_kw):
    """Median device ms per run_frames step (preallocated outputs, points on) for each dtype, alternated."""
    setups = {}
    for name, dt in DTYPES:
        pipe = LineEndPipeline(zoom_ratio=SCALE, out_dtype=dt, **pipe_kw)
        res = pipe.run_frames(frames)   # plan, workspace and the output shapes
        n = int(res.orient.shape[0])
        bufs = (torch.empty_like(res.orient), torch.empty_like(res.padded_line_end),
                torch.empty((64 * n, 4), dtype=torch.int64, device=frames.device),
                torch.zeros(1, dtype=torch.int64, device=frames.device))
        fn = (lambda p, b: lambda: p.run_frames(frames, out=b))(pipe, bufs)
        time_device(fn, 3)
        setups[name] = (fn, res.orient.element_size() * res.orient.numel() * 2)
    times = {name: [] for name, _ in DTYPES}
    for _ in range(runs):
        for name, _ in DTYPES:
            times[name].append(time_device(setups[name][0], steps))
    return {name: dict(summary(times[name]), output_bytes_per_step=setups[name][1]) for name, _ in DTYPES}


def link_probe(dev):
    """bench.py's e2e.link probe: 256 MiB pinned H2D and D2H copies at once, GB/s per direction."""
    nbytes = 256 << 20
    h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_in = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_out = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def both():
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)

    both()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(4):
        both()
    torch.cuda.synchronize()
    return nbytes / ((time.perf_counter() - t0) / 4) / 1e9


def e2e(host_frames, runs, steps, dev):
    b = host_frames.shape[0]
    setups = {}
    for name, dt in DTYPES:
        pipe = LineEndPipeline(zoom_ratio=SCALE, out_dtype=dt)
        res = pipe.run_host(host_frames)
        np_dt = np.float16 if dt == torch.float16 else np.float32
        o = torch.empty(res.orient.shape, dtype=dt).pin_memory().numpy()
        e = torch.empty(res.orient.shape, dtype=dt).pin_memory().numpy()
        assert o.dtype == np_dt
        fn = (lambda p, o, e: lambda: p.run_host(host_frames, o, e))(pipe, o, e)
        fn()
        setups[name] = (fn, o.nbytes + e.nbytes)
    h2d = host_frames.nbytes
    out = {}
    ms = {name: [] for name, _ in DTYPES}
    probes = []
    for _ in range(runs):
        for name, _ in DTYPES:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                setups[name][0]()
            torch.cuda.synchronize()
            ms[name].append((time.perf_counter() - t0) * 1000.0 / steps)
        probes.append(link_probe(dev))
    probe = statistics.median(probes)
    for name, _ in DTYPES:
        d2h = setups[name][1]
        med = statistics.median(ms[name])
        out[name] = {"ms_per_step": summary(ms[name]), "frames_per_s": b / (med * 1e-3),
                     "frames_per_s_range": [b / (max(ms[name]) * 1e-3), b / (min(ms[name]) * 1e-3)],
                     "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                     "larger_direction_gbs": max(h2d, d2h) / (med * 1e-3) / 1e9,
                     "frac_of_probe": max(h2d, d2h) / (med * 1e-3) / 1e9 / probe}
    out["link_probe_gbs_each_way"] = summary(probes)
    out["float16_speedup"] = statistics.median(ms["float32"]) / statistics.median(ms["float16"])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=8)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--e2e-steps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "half_bench.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    record = {"card": card(), "runs_per_dtype": args.runs, "alternated": True}
    rs = np.random.RandomState(3000)
    host_c3 = torch.from_numpy(rs.randint(0, 256, size=(64, 1080, 1920, 3), dtype=np.uint8)).pin_memory()
    c3 = host_c3.to(dev)
    record["c3"] = {"workload": "64 x 1080p uint8, scale sqrt2, 6 levels, run_frames with points (device ms per step)",
                    "steps_per_run": args.steps, **device_steps(c3, args.runs, args.steps)}
    del c3
    c4 = torch.from_numpy(rs.randint(0, 256, size=(16, 2160, 3840, 3), dtype=np.uint8)).to(dev)
    record["c4"] = {"workload": "16 x 3840x2160 uint8, scale sqrt2, 8 levels, run_frames with points (device ms per step)",
                    "steps_per_run": args.steps}
    for nb in (4, 8, 12, 16):
        record["c4"]["orientations_%d" % nb] = device_steps(c4, args.runs, args.steps, orientations=nb)
    del c4
    torch.cuda.empty_cache()
    record["e2e"] = {"workload": "run_host, 64 x 1080p uint8 from page-locked host memory into page-locked outputs, "
                                 "scale sqrt2, 6 levels", "steps_per_run": args.e2e_steps,
                     **e2e(host_c3.numpy(), args.runs, args.e2e_steps, dev)}
    record["card_after"] = card()
    with open(args.out, "w") as f:
        json.dump(record, f, indent=1)
    c3r = record["c3"]
    print("c3 ms: f32 %.4f f16 %.4f" % (c3r["float32"]["median"], c3r["float16"]["median"]))
    for nb in (4, 8, 12, 16):
        r = record["c4"]["orientations_%d" % nb]
        print("c4 nb=%d ms: f32 %.4f f16 %.4f" % (nb, r["float32"]["median"], r["float16"]["median"]))
    e = record["e2e"]
    print("e2e fps: f32 %.0f (%.3f of probe) f16 %.0f (%.3f of probe), x%.3f" % (
        e["float32"]["frames_per_s"], e["float32"]["frac_of_probe"], e["float16"]["frames_per_s"],
        e["float16"]["frac_of_probe"], e["float16_speedup"]))


if __name__ == "__main__":
    main()
