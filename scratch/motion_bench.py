"""Frame-to-frame motion: what the three motion kernels take, the pan they recover from a panned scene with the inlier
shares at several thresholds and hypothesis counts, and what motion costs on top of the matches end to end.

  input    64 x 1080p BGR uint8 frames, each a crop of one seeded texture moved by PAN = (dy, dx) pixels per frame
           (matches_bench.py's scene), so the true motion of every pair is T = [I | -PAN]. float32 outputs,
           3 orientations, scale sqrt2 (6 levels). Matches: patch radius 2, search radius 8, max_ratio 0.64.
  motion   for peaks p = 0.1, 0.5 and 0.9, on the records and matches of run_frames_matches: for thresholds 1, 2, 4
           and 8 frame pixels and 64, 256 and 1024 hypotheses, the largest |T - truth| over the 63 pairs (linear part
           and translation) and the inlier share (inlier_count / matched; min, median, max over the pairs).
  kernels  silent_estimate_motion alone at 256 and 1024 hypotheses (threshold 2): the three kernels together per call
           from CUDA events around LAUNCHES back-to-back calls, and each kernel's duration from torch.profiler in a run
           of its own (median over LAUNCHES launches, per run). They are programmatic dependent launches, so a later
           kernel's profiler duration can include its wait for the one before; the events give the cost of a call.
  e2e      run_frames_motion against run_frames_matches (device frames) and run_host_motion against run_host_matches
           (page-locked host frames), the defaults of threshold and hypotheses, alternated, host clock around calls
           that synchronise.

The card's name and power limit are read in the same process. Writes one JSON file (--out).

    python scratch/motion_bench.py --out motion_bench.json [--runs 5]
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
from matches_bench import PAN, SCALE, panned_frames   # noqa: E402
from pysilent_b200 import LineEndPipeline, _ops   # noqa: E402

PERCENTS = (0.1, 0.5, 0.9)
R_PATCH, R_SEARCH, RATIO = 2, 8, 0.64
THRESHOLDS = (1.0, 2.0, 4.0, 8.0)
HYPOTHESES = (64, 256, 1024)
KERNELS = ("motion_compact_kernel", "motion_score_kernel", "motion_refine_kernel")
LAUNCHES = 20
TRUTH = np.array([[1.0, 0.0, -PAN[0]], [0.0, 1.0, -PAN[1]]])


def profiled(fn):
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


def accuracy(mo):
    """Errors over the pairs that have a model (p = 0.1 leaves some pairs under 3 correspondences)."""
    T, n, m = (t.cpu().numpy() for t in mo[:3])
    fit = ~np.isnan(T).any(axis=(1, 2))
    T, n, m = T[fit], n[fit], m[fit]
    share = n / np.maximum(m, 1)
    return {"pairs_with_a_model": int(fit.sum()),
            "max_abs_linear_error": float(np.abs(T[:, :, :2] - TRUTH[:, :2]).max()),
            "max_abs_shift_error_px": float(np.abs(T[:, :, 2] - TRUTH[:, 2]).max()),
            "mean_shift": [float(v) for v in T[:, :, 2].mean(axis=0)],
            "inlier_share": {"min": float(share.min()), "median": float(np.median(share)), "max": float(share.max())},
            "matched": {"min": int(m.min()), "max": int(m.max())}}


def motion(frames, runs):
    res = {}
    for p in PERCENTS:
        pipe = LineEndPipeline(zoom_ratio=SCALE, peaks=p)
        rec, m = pipe.run_frames_matches(frames, R_PATCH, R_SEARCH, RATIO)
        k = len(rec.points)
        count = torch.full((1,), k, dtype=torch.int64, device=frames.device)
        args = (rec.frame_offsets, rec.frame_yx, m.next, count)
        entry = {"points": k, "matches": int((m.next >= 0).sum())}
        for thr in THRESHOLDS:
            for h in HYPOTHESES:
                entry["threshold=%g hypotheses=%d" % (thr, h)] = accuracy(_ops.estimate_motion(*args, h, thr, 0))
        pairs = len(rec.frame_offsets) - 2
        dev = frames.device
        outs = dict(transform=torch.empty((pairs, 2, 3), dtype=torch.float64, device=dev),
                    inlier_count=torch.empty(pairs, dtype=torch.int64, device=dev),
                    matched=torch.empty(pairs, dtype=torch.int64, device=dev),
                    inlier=torch.empty(k, dtype=torch.uint8, device=dev),
                    workspace=torch.empty(_ops.motion_workspace_bytes(k), dtype=torch.uint8, device=dev))
        for h in (256, 1024):
            fn = (lambda h: lambda: _ops.estimate_motion(*args, h, 2.0, 0, **outs))(h)
            for _ in range(5):
                fn()
            torch.cuda.synchronize()
            events = [time_device(fn, LAUNCHES) * 1000.0 for _ in range(runs)]
            per = [profiled(fn) for _ in range(runs)]
            entry["kernels hypotheses=%d" % h] = {
                "events_us_per_call": summary(events),
                "profiler_kernel_us_median": {kk: statistics.median(x[kk] for x in per) for kk in KERNELS},
                "per_run": per}
        res["p=%g" % p] = entry
        del rec, m, args, outs
        torch.cuda.empty_cache()
    return res


def alternate(arms, runs, steps):
    for fn in arms.values():
        fn()
    ms = {k: [] for k in arms}
    for _ in range(runs):
        for k, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
            ms[k].append((time.perf_counter() - t0) * 1000.0 / steps)
    return {k: {"ms_per_call": summary(v)} for k, v in ms.items()}


def e2e(frames, bgr, runs, steps):
    arms = {}
    for p in PERCENTS:
        pipe = LineEndPipeline(zoom_ratio=SCALE, peaks=p)
        arms["run_frames_motion p=%g" % p] = (lambda pipe: lambda: pipe.run_frames_motion(
            frames, R_PATCH, R_SEARCH, RATIO))(pipe)
        arms["run_frames_matches p=%g" % p] = (lambda pipe: lambda: pipe.run_frames_matches(
            frames, R_PATCH, R_SEARCH, RATIO))(pipe)
        arms["run_host_motion p=%g" % p] = (lambda pipe: lambda: pipe.run_host_motion(
            bgr, R_PATCH, R_SEARCH, RATIO))(pipe)
        arms["run_host_matches p=%g" % p] = (lambda pipe: lambda: pipe.run_host_matches(
            bgr, R_PATCH, R_SEARCH, RATIO))(pipe)
    return alternate(arms, runs, steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "motion_bench.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    record = {"card": card(), "runs": args.runs, "launches_per_run": LAUNCHES, "pan_dy_dx": PAN,
              "truth": TRUTH.tolist()}
    host = torch.empty((64, 1080, 1920, 3), dtype=torch.uint8, pin_memory=True)
    host.numpy()[...] = panned_frames(4000, 64, 1080, 1920, PAN)
    frames = host.to(dev)
    record["motion"] = {"workload": "64 x 1080p BGR uint8 panned by %s per frame, scale sqrt2, 6 levels, 3 "
                                    "orientations, float32 outputs, matches r=%d R=%d max_ratio=%g"
                                    % (PAN, R_PATCH, R_SEARCH, RATIO), **motion(frames, args.runs)}
    torch.cuda.empty_cache()
    record["e2e"] = {"workload": "the same frames and matches, default threshold and hypotheses", "steps_per_run": 2,
                     **e2e(frames, host.numpy(), args.runs, 2)}
    record["card_after"] = card()
    with open(args.out, "w") as f:
        json.dump(record, f, indent=1)
    print(json.dumps(record["card"]))
    for k, v in record["motion"].items():
        if not isinstance(v, dict):
            continue
        print("%s: %d points, %d matches" % (k, v["points"], v["matches"]))
        for kk, a in v.items():
            if kk.startswith("threshold"):
                print("  %s: %d pairs, |dA| %.5f |dt| %.4f share %.4f/%.4f/%.4f" % (
                    kk, a["pairs_with_a_model"], a["max_abs_linear_error"], a["max_abs_shift_error_px"], a["inlier_share"]["min"],
                    a["inlier_share"]["median"], a["inlier_share"]["max"]))
            elif kk.startswith("kernels"):
                print("  %s: %s, call %.2f us (events)" % (kk, ", ".join(
                    "%s %.2f us" % (n.replace("_kernel", ""), t) for n, t in a["profiler_kernel_us_median"].items()),
                    a["events_us_per_call"]["median"]))
    for arm, v in record["e2e"].items():
        if isinstance(v, dict):
            m = v["ms_per_call"]
            print("e2e %s: %.3f ms [%.3f-%.3f]" % (arm, m["median"], m["min"], m["max"]))


if __name__ == "__main__":
    main()
