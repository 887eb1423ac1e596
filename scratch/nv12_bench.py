"""BGR against NV12 frames (LineEndPipeline(frame_format=...)), alternated in one process, on four workloads:

  conv    silent_nv12_to_bgr alone on 64 x 1080p frames (device ms per call), and the GB/s it reaches on its own bytes
          (NV12 read + BGR written)
  c3      device step (ms) of run_frames with points: 64 x 1080p, scale sqrt2, 6 levels (BASELINE C3), float32 and
          float16 outputs
  c4      device step (ms) of run_frames on C4's frames (16 x 3840x2160, scale sqrt2, 8 levels), bank of 8
  e2e     run_host on the 64 x 1080p frames from page-locked host buffers (frames/s), float32 and float16 outputs,
          beside the concurrent pinned H2D + D2H copy probe of bench.py's e2e.link

The BGR frames are the NV12 frames converted, so both arms see the same images. Each measurement is repeated --runs
times per arm, the arms alternating; medians and ranges are reported. The card's name and power limit are read in the
same process. Writes one JSON file (--out).

    python scratch/nv12_bench.py --out nv12_bench.json [--runs 8] [--steps 20]
"""
import argparse
import ctypes
import json
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scratch"))
from half_bench import SCALE, card, link_probe, summary, time_device   # noqa: E402
from pysilent_b200 import LineEndPipeline, _lib, _ops   # noqa: E402


def alternate(setups, runs, measure):
    """measure(fn) for every arm of ``setups`` ({name: fn}), ``runs`` rounds with the arms alternating."""
    times = {name: [] for name in setups}
    for _ in range(runs):
        for name, fn in setups.items():
            times[name].append(measure(fn))
    return times


def step_fn(frames, fmt, **pipe_kw):
    """run_frames with preallocated outputs and points on, for frames in format ``fmt``."""
    pipe = LineEndPipeline(zoom_ratio=SCALE, frame_format=fmt, **pipe_kw)
    res = pipe.run_frames(frames)   # plan, workspace and the output shapes
    n = int(res.orient.shape[0])
    bufs = (torch.empty_like(res.orient), torch.empty_like(res.padded_line_end),
            torch.empty((64 * n, 4), dtype=torch.int64, device=frames.device),
            torch.zeros(1, dtype=torch.int64, device=frames.device))
    fn = lambda: pipe.run_frames(frames, out=bufs)   # noqa: E731
    time_device(fn, 3)
    return fn


def device_steps(arms, runs, steps):
    """arms: {name: fn}; median device ms per step of each, alternated."""
    times = alternate(arms, runs, lambda fn: time_device(fn, steps))
    out = {name: summary(t) for name, t in times.items()}
    return out


def conversion(nv12, runs, steps):
    b, rows, w = (int(v) for v in nv12.shape)
    h = 2 * rows // 3
    bgr = torch.empty((b, h, w, 3), dtype=torch.uint8, device=nv12.device)
    lib = _lib.lib()

    def fn():
        _lib.check(lib.silent_nv12_to_bgr(_ops.ptr(nv12), b, h, w, _ops.ptr(bgr), _ops.stream_ptr()))
    time_device(fn, 3)
    times = alternate({"nv12_to_bgr": fn}, runs, lambda f: time_device(f, steps))["nv12_to_bgr"]
    nbytes = nv12.numel() + bgr.numel()
    med = statistics.median(times)
    return {"ms_per_call": summary(times), "bytes_per_call": nbytes, "gbs": nbytes / (med * 1e-3) / 1e9,
            "gbs_range": [nbytes / (max(times) * 1e-3) / 1e9, nbytes / (min(times) * 1e-3) / 1e9]}


def e2e(host, runs, steps, dev):
    """host: {fmt: page-locked numpy frames}; run_host frames/s per (format, output dtype), alternated."""
    setups, sizes = {}, {}
    for out_name, dt in (("float32", torch.float32), ("float16", torch.float16)):
        for fmt, frames in host.items():
            pipe = LineEndPipeline(zoom_ratio=SCALE, out_dtype=dt, frame_format=fmt)
            res = pipe.run_host(frames)
            o = torch.empty(res.orient.shape, dtype=dt).pin_memory().numpy()
            e = torch.empty(res.orient.shape, dtype=dt).pin_memory().numpy()
            fn = (lambda p, f, o, e: lambda: p.run_host(f, o, e))(pipe, frames, o, e)
            fn()
            name = "%s_%s" % (fmt, out_name)
            setups[name], sizes[name] = fn, (frames.nbytes, o.nbytes + e.nbytes)

    import time

    def measure(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1000.0 / steps

    ms = {name: [] for name in setups}
    probes = []
    for _ in range(runs):
        for name, fn in setups.items():
            ms[name].append(measure(fn))
        probes.append(link_probe(dev))
    probe = statistics.median(probes)
    b = next(iter(host.values())).shape[0]
    out = {"link_probe_gbs_each_way": summary(probes)}
    for name in setups:
        h2d, d2h = sizes[name]
        med = statistics.median(ms[name])
        out[name] = {"ms_per_step": summary(ms[name]), "frames_per_s": b / (med * 1e-3),
                     "frames_per_s_range": [b / (max(ms[name]) * 1e-3), b / (min(ms[name]) * 1e-3)],
                     "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                     "frac_of_probe": max(h2d, d2h) / (med * 1e-3) / 1e9 / probe}
    for o in ("float32", "float16"):
        out["nv12_speedup_%s" % o] = statistics.median(ms["bgr_" + o]) / statistics.median(ms["nv12_" + o])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=8)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--e2e-steps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "nv12_bench.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    record = {"card": card(), "runs_per_arm": args.runs, "alternated": True}
    rs = np.random.RandomState(3100)
    nv12_c3 = torch.from_numpy(rs.randint(0, 256, size=(64, 1620, 1920), dtype=np.uint8)).to(dev)
    bgr_c3 = _ops.nv12_to_bgr(nv12_c3)
    record["conv"] = {"workload": "silent_nv12_to_bgr, 64 x 1080p, whole frames (device ms per call)",
                      "steps_per_run": args.steps, **conversion(nv12_c3, args.runs, args.steps)}
    arms = {}
    for out_name, dt in (("float32", torch.float32), ("float16", torch.float16)):
        arms["bgr_" + out_name] = step_fn(bgr_c3, "bgr", out_dtype=dt)
        arms["nv12_" + out_name] = step_fn(nv12_c3, "nv12", out_dtype=dt)
    record["c3"] = {"workload": "64 x 1080p, scale sqrt2, 6 levels, run_frames with points (device ms per step)",
                    "steps_per_run": args.steps, **device_steps(arms, args.runs, args.steps)}
    host = {"bgr": torch.from_numpy(bgr_c3.cpu().numpy()).pin_memory().numpy(),
            "nv12": torch.from_numpy(nv12_c3.cpu().numpy()).pin_memory().numpy()}
    del arms, nv12_c3, bgr_c3
    torch.cuda.empty_cache()
    nv12_c4 = torch.from_numpy(rs.randint(0, 256, size=(16, 3240, 3840), dtype=np.uint8)).to(dev)
    bgr_c4 = _ops.nv12_to_bgr(nv12_c4)
    arms = {"bgr": step_fn(bgr_c4, "bgr", orientations=8), "nv12": step_fn(nv12_c4, "nv12", orientations=8)}
    record["c4_bank8"] = {"workload": "16 x 3840x2160, scale sqrt2, 8 levels, bank of 8, run_frames with points "
                                      "(device ms per step)", "steps_per_run": args.steps,
                          **device_steps(arms, args.runs, args.steps)}
    del arms, nv12_c4, bgr_c4
    torch.cuda.empty_cache()
    record["e2e"] = {"workload": "run_host, 64 x 1080p from page-locked host memory into page-locked outputs, "
                                 "scale sqrt2, 6 levels", "steps_per_run": args.e2e_steps,
                     **e2e(host, args.runs, args.e2e_steps, dev)}
    record["card_after"] = card()
    with open(args.out, "w") as f:
        json.dump(record, f, indent=1)
    c = record["conv"]
    print("conv ms %.4f (%.0f GB/s)" % (c["ms_per_call"]["median"], c["gbs"]))
    for k in ("bgr_float32", "nv12_float32", "bgr_float16", "nv12_float16"):
        print("c3 %s ms %.4f" % (k, record["c3"][k]["median"]))
    print("c4 bank8 ms: bgr %.4f nv12 %.4f" % (record["c4_bank8"]["bgr"]["median"], record["c4_bank8"]["nv12"]["median"]))
    e = record["e2e"]
    for k in ("bgr_float32", "nv12_float32", "bgr_float16", "nv12_float16"):
        print("e2e %s fps %.0f (%.3f of probe)" % (k, e[k]["frames_per_s"], e[k]["frac_of_probe"]))


if __name__ == "__main__":
    main()
