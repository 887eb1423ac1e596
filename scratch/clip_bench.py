"""LineEndDisplayer over a clip: 64 consecutive device-resident 1080p frames of one camera (zoom_ratio = sqrt(2), 6
levels), run as 64 x run_frames_display (pipeline + display_tensors per frame) against one run_clip; and the display
recurrence alone, 64 silent_display_tensors calls against one silent_display_sequence on the same gray levels.

    python scratch/clip_bench.py [--reps 20] [--out clip_bench.json]

Prints and writes one JSON object: device and wall ms per frame of each arm (median over reps, with the range), the
kernel times from a separate torch.profiler run, and display_sequence_kernel's launch shape (grid / block / shared memory
from the trace, registers and spills from ptxas.log of the build)."""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pysilent_b200 import LineEndDisplayer, _ops   # noqa: E402
from pysilent_b200.util.color import get_value_from_color   # noqa: E402

T, H, W = 64, 1080, 1920


def timed(fn, reps):
    """Median and range of device ms (events) and wall ms (host clock to a synchronise) of fn over reps runs."""
    dev, wall = [], []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(a.elapsed_time(b))
    return dict(device_ms=float(np.median(dev)), device_ms_range=[float(min(dev)), float(max(dev))],
                wall_ms=float(np.median(wall)), wall_ms_range=[float(min(wall)), float(max(wall))])


def per_frame(r):
    return {k.replace("_ms", "_ms_per_frame"): (v / T if not isinstance(v, list) else [x / T for x in v])
            for k, v in r.items()}


def kernel_profile(fn):
    """Kernel name -> (total ms, launches, first event's args) of one call of fn under torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    path = os.path.join(tempfile.mkdtemp(), "trace.json")
    prof.export_chrome_trace(path)
    out = {}
    for ev in json.load(open(path))["traceEvents"]:
        if ev.get("cat") != "kernel":
            continue
        name = re.sub(r"\(.*", "", ev["name"]).replace("void ", "")
        ms, k, args = out.get(name, (0.0, 0, ev.get("args", {})))
        out[name] = (ms + ev["dur"] / 1e3, k + 1, args)
    return out


def ptxas_properties(kernel):
    log = os.path.join(ROOT, "pysilent_b200", "build", "ptxas.log")
    if not os.path.exists(log):
        return "ptxas.log missing"
    text = open(log).read()
    res = {}
    for m in re.finditer(r"Function properties for (\S*%s\S*)\n\s*(.*)\nptxas info\s*: (Used .*)" % kernel, text):
        res[m.group(1)] = m.group(2).strip() + "; " + m.group(3).strip()
    return res


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:   # the measurement stands without it; say so in the record
        return "unavailable: %s" % exc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "clip_bench needs a CUDA device"
    frames = torch.from_numpy(np.random.RandomState(7).randint(0, 256, size=(T, H, W, 3), dtype=np.uint8)).cuda()

    step_disp, clip_disp = LineEndDisplayer(zoom_ratio=2 ** .5), LineEndDisplayer(zoom_ratio=2 ** .5)

    def per_step():
        for t in range(T):
            step_disp.run_frames_display(frames[t])

    def clip():
        clip_disp.run_clip(frames)

    # warm-up (plans, allocator, module loads), then the two arms alternated rep by rep
    per_step()
    clip()
    a_runs, b_runs = [], []
    for _ in range(args.reps):
        a_runs.append(timed(per_step, 1))
        b_runs.append(timed(clip, 1))

    def summary(runs):
        d = [r["device_ms"] for r in runs]
        w = [r["wall_ms"] for r in runs]
        return dict(device_ms=float(np.median(d)), device_ms_range=[min(d), max(d)], wall_ms=float(np.median(w)),
                    wall_ms_range=[min(w), max(w)])
    per_step_r, clip_r = summary(a_runs), summary(b_runs)
    same = bool(torch.equal(step_disp.energy_values.nan_to_num(123.0), clip_disp.energy_values.nan_to_num(123.0)))

    # the recurrence alone on the gray levels of the clip
    res = clip_disp.run_frames(frames, want_points=False)
    gray = get_value_from_color(res.padded_line_end)
    n = gray.shape[0] // T
    e1 = torch.full((n, 64, 96, 1), 8.0, device="cuda")
    e2 = e1.clone()

    def tensors_loop():
        for t in range(T):
            _ops.display_tensors(gray[t * n:(t + 1) * n], e1, 3, 3, 116, 174, 1, 1, 1)

    def sequence():
        _ops.display_sequence(gray, e2, T, 3, 3, 116, 174, 1, 1, 1)

    tensors_loop()
    sequence()
    loop_r = timed(tensors_loop, args.reps)
    seq_r = timed(sequence, args.reps)
    prof_seq = kernel_profile(sequence)
    prof_loop = kernel_profile(tensors_loop)
    seq_kernel = [(k, v) for k, v in prof_seq.items() if "display_sequence_kernel" in k]
    launch = {}
    if seq_kernel:
        name, (ms, cnt, kargs) = seq_kernel[0]
        grid = kargs.get("grid", [0])
        launch = dict(kernel=name, grid=grid, block=kargs.get("block"), dynamic_shared_bytes=kargs.get("shared memory"),
                      registers_per_thread=kargs.get("registers per thread"),
                      cluster_size=(grid[0] // n if grid and grid[0] else None), slices=n)

    out = dict(
        workload="LineEndDisplayer, %d consecutive %dx%d uint8 frames of one camera, device-resident, zoom_ratio=sqrt(2) "
                 "(%d levels of 192x288, 64x96 boosting cells per level)" % (T, H, W, n),
        gpu=gpu_info(), reps=args.reps,
        per_step=dict(what="%d x run_frames_display(frames[t]) (pipeline + display_tensors, 2 display launches)" % T,
                      **per_frame(per_step_r)),
        run_clip=dict(what="one run_clip(frames) (pipeline over %d frames + display_sequence)" % T, **per_frame(clip_r)),
        run_clip_speedup_device=per_step_r["device_ms"] / clip_r["device_ms"],
        run_clip_speedup_wall=per_step_r["wall_ms"] / clip_r["wall_ms"],
        final_energy_equal=same,
        recurrence=dict(
            what="display chain alone on the clip's %d gray levels: %d x silent_display_tensors vs one "
                 "silent_display_sequence" % (T * n, T),
            display_tensors_loop=per_frame(loop_r), display_sequence=per_frame(seq_r),
            kernels_display_sequence={k: dict(ms=v[0], launches=v[1]) for k, v in prof_seq.items()},
            kernels_display_tensors_loop={k: dict(ms=v[0], launches=v[1]) for k, v in prof_loop.items()}),
        display_sequence_kernel=dict(launch=launch, ptxas=ptxas_properties("display_sequence_kernel")),
    )
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
