"""Config C4's workload (16 x 3840x2160 uint8 frames, scale sqrt2 -> 8 levels) through the fused orientation bank at
4, 8, 12 and 16 orientations: frames/s, algorithmic bytes per frame, fraction of the project's HBM denominator, and the
per-stage device times of silent_plan_stage_ms / silent_plan_stack_split_ms (stack_b = stack_bank_kernel). At n = 8 the
old entry (silent_pipeline_run_bank) and the new one (silent_pipeline_run_orientations) are timed alternately in the same
process. Writes one JSON file (--out).

    python scratch/bank_bench.py --out bank_bench.json [--widths 4,8,12,16] [--steps 50]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pysilent_b200 import LineEndPipeline, _lib, _ops   # noqa: E402

PEAK_GBS = 6541.8   # the project's HBM denominator (bench.py)
BATCH, SCALE = 16, 2 ** .5


def card():
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                    text=True).splitlines()[torch.cuda.current_device()]
        name, power, clock = (v.strip() for v in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:   # the numbers stay valid; the record says why the card line is missing
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % exc}


def time_steps(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def stage_times(plan, fn, steps):
    """Median per-stage device times (ms) over `steps` runs with the plan's timing events on."""
    L = _lib.lib()
    _lib.check(L.silent_plan_enable_timing(plan.handle, 1))
    rows = []
    for _ in range(steps):
        fn()
        v = [ctypes.c_float() for _ in range(5)]
        _lib.check(L.silent_plan_stage_ms(plan.handle, *[ctypes.byref(x) for x in v[:3]]))
        _lib.check(L.silent_plan_stack_split_ms(plan.handle, *[ctypes.byref(x) for x in v[3:]]))
        rows.append([x.value for x in v])
    _lib.check(L.silent_plan_enable_timing(plan.handle, 0))
    keys = ("pyramid_ms", "stack_ms", "emit_ms", "stack_a_ms", "stack_bank_kernel_ms")
    return {k: statistics.median(r[i] for r in rows) for i, k in enumerate(keys)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--widths", default="4,8,12,16")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5, help="alternations of the old and new n = 8 entry")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bank_bench measures the B200; there is no CPU arm"
    dev = torch.device("cuda", torch.cuda.current_device())
    frames = torch.from_numpy(np.random.RandomState(4).randint(0, 256, size=(BATCH, 2160, 3840, 3), dtype=np.uint8)).to(dev)
    result = {"workload": "C4 frames: %d x 3840x2160 uint8, scale sqrt2" % BATCH, "card": card(), "steps": args.steps,
              "peak_gbs": PEAK_GBS, "widths": {}}
    for n in (int(v) for v in args.widths.split(",")):
        pipe = LineEndPipeline(zoom_ratio=SCALE, orientations=n)
        fn = lambda: pipe.run_frames(frames)   # noqa: E731  (as bench.py runs C4: points included, one count sync)
        for _ in range(3):
            res = fn()
        plan = pipe.plan_for(frames)
        levels = plan.levels
        crop = plan.algorithmic_bytes - 2 * levels * plan.h * plan.w * 3 * 4
        alg = crop + 2 * levels * plan.h * plan.w * n * 4
        ms = time_steps(fn, args.steps)
        fps = BATCH / (ms * 1e-3)
        entry = {"levels": levels, "ms_per_step": ms, "frames_per_s": fps, "algorithmic_bytes_per_frame": int(alg),
                 "achieved_gbs": alg * fps / 1e9, "frac_of_peak": alg * fps / 1e9 / PEAK_GBS, "points": len(res.points)}
        entry.update(stage_times(plan, fn, args.steps))
        result["widths"][str(n)] = entry
        print("n=%2d: %.3f ms/step, %.0f frames/s, %.1f MB/frame, %.3f of %.1f GB/s, stack_bank_kernel %.3f ms" % (
            n, ms, fps, alg / 1e6, entry["frac_of_peak"], PEAK_GBS, entry["stack_bank_kernel_ms"]), flush=True)
        if n == 8:
            result["n8_entries"] = entries_alternated(pipe, plan, frames, args.steps, args.rounds)
        del res
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result.get("n8_entries", {})))


def entries_alternated(pipe, plan, frames, steps, rounds):
    """Device time per step of silent_pipeline_run_bank and silent_pipeline_run_orientations, alternated, preallocated
    outputs, no host synchronisation inside the timed window."""
    L = _lib.lib()
    n = BATCH * plan.levels
    f = pipe.bank_filters()
    old = _lib.make_bank_weights(f["rgc"], f["rgby"], f["stripe"], f["blur"], f["end"])
    new = pipe.orientation_bank()
    o = torch.empty((n, plan.h, plan.w, 8), dtype=torch.float32, device=frames.device)
    l, cap = torch.empty_like(o), 64 * n
    pts = torch.empty((cap, 4), dtype=torch.int64, device=frames.device)
    cnt = torch.zeros(1, dtype=torch.int64, device=frames.device)
    calls = {"silent_pipeline_run_bank": (L.silent_pipeline_run_bank, old),
             "silent_pipeline_run_orientations": (L.silent_pipeline_run_orientations, new)}
    times = {k: [] for k in calls}
    for r in range(rounds + 1):
        for name, (fn, w) in calls.items():
            ms = time_steps(lambda: _lib.check(fn(plan.handle, ctypes.byref(w), _ops.ptr(frames), BATCH, _ops.ptr(o),
                                                  _ops.ptr(l), _ops.ptr(pts), cap, _ops.ptr(cnt), _ops.stream_ptr())),
                            steps)
            if r:   # round 0 warms both up
                times[name].append(ms)
    return {k: {"ms_per_step": v, "median_frames_per_s": BATCH / (statistics.median(v) * 1e-3)} for k, v in times.items()}


if __name__ == "__main__":
    main()
