"""Feature-point matches: how many points of a panned scene find their twin in the next frame, how many of those agree
with the pan, what the two match kernels take, and what matching costs run_host_records end to end.

  input    64 x 1080p BGR uint8 frames, each a crop of one seeded texture (blurred noise, larger than the frame) moved by
           PAN = (dy, dx) pixels per frame, so frame f + 1 shows frame f's content shifted by -PAN: true correspondences
           exist at every level. float32 outputs, 3 orientations, scale sqrt2 (6 levels).
  matches  for peaks p = 0.1 and 0.5, patch radius r = 2 and 4, search radius R = 8 and 16, and max_ratio 1 and 0.64:
           the points, the accepted matches, and the share of matches whose frame_yx displacement is -PAN within one
           level pixel of that level (the level's largest frame-coordinate step per axis).
  kernels  silent_match_points alone on the records of each (p, r, R), max_ratio 0.64: the two kernels together per
           call from CUDA events around LAUNCHES back-to-back calls, and each kernel's duration from torch.profiler in a
           run of its own (median over LAUNCHES launches, per run). Both are programmatic dependent launches, so
           match_finalise_kernel's CTAs start while match_search_kernel drains and wait for it: its profiler duration
           includes that wait and overlaps the search's; the events give the cost of a call.
  e2e      run_host_matches(r = 4, R = 16, max_ratio 0.64) against run_host_records() (the same records without patches)
           and run_host_records(patch_radius=4) (the patches downloaded), p = 0.1 and 0.5, page-locked frames,
           alternated, host clock around calls that synchronise.

The card's name and power limit are read in the same process. Writes one JSON file (--out).

    python scratch/matches_bench.py --out matches_bench.json [--runs 5]
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
PAN = (3, -5)
PERCENTS = (0.1, 0.5)
PATCH_RADII = (2, 4)
SEARCH_RADII = (8, 16)
RATIOS = (1.0, 0.64)
KERNELS = ("match_search_kernel", "match_finalise_kernel")
LAUNCHES = 20


def panned_frames(seed, batch, h, w, pan):
    """``batch`` crops of one texture of blurred uniform noise, frame f at offset f * pan."""
    from scipy.ndimage import gaussian_filter
    dy, dx = pan
    H, W = h + abs(dy) * batch + 8, w + abs(dx) * batch + 8
    tex = gaussian_filter(np.random.RandomState(seed).rand(H, W, 3).astype(np.float32), (1.5, 1.5, 0))
    tex = np.clip((tex - tex.mean()) / tex.std() * 60 + 128, 0, 255).astype(np.uint8)
    y0 = 4 if dy >= 0 else H - h - 4
    x0 = 4 if dx >= 0 else W - w - 4
    return np.stack([tex[y0 + f * dy: y0 + f * dy + h, x0 + f * dx: x0 + f * dx + w] for f in range(batch)])


def pan_agreement(pts, frame_yx, nxt, plan, pan):
    """(share of accepted matches whose displacement is -pan within one level pixel, accepted matches)."""
    i = np.nonzero(nxt >= 0)[0]
    if len(i) == 0:
        return 0.0, 0
    lvl = pts[i, 0] % plan.levels
    step = np.array([[np.nanmax(np.diff(c)) for c in plan.level_coords(l)] for l in range(plan.levels)])[lvl]
    d = frame_yx[nxt[i]] - frame_yx[i]
    ok = (np.abs(d[:, 0] + pan[0]) <= step[:, 0]) & (np.abs(d[:, 1] + pan[1]) <= step[:, 1])
    return float(ok.mean()), len(i)


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


def matches(frames, runs):
    res = {}
    for p in PERCENTS:
        pipe = LineEndPipeline(zoom_ratio=SCALE, peaks=p)
        plan = pipe.plan_for(frames)
        for r in PATCH_RADII:
            _, (pts, _, yx, values) = pipe._record_rows(frames, None, None, r)   # run_frames_records' rows
            k = len(pts)
            count = torch.full((1,), k, dtype=torch.int64, device=frames.device)
            outs = [torch.empty(k, dtype=torch.int64, device=frames.device) for _ in range(2)] + \
                [torch.empty(k, device=frames.device)]
            for R in SEARCH_RADII:
                entry = {"points": k, "descriptor_floats": int(values[0].numel())}
                for ratio in RATIOS:
                    nxt = _ops.match_points(pts, count, values, plan.levels, R, ratio, *outs)[0]
                    share, n = pan_agreement(pts.cpu().numpy(), yx.cpu().numpy(), nxt.cpu().numpy(), plan, PAN)
                    entry["max_ratio=%g" % ratio] = {"matches": n, "matches_per_point": n / k, "agree_with_pan": share}
                fn = lambda: _ops.match_points(pts, count, values, plan.levels, R, 0.64, *outs)  # noqa: E731
                for _ in range(5):
                    fn()
                torch.cuda.synchronize()
                events = [time_device(fn, LAUNCHES) * 1000.0 for _ in range(runs)]
                entry["events_us_per_call"] = summary(events)
                per = [profiled(fn) for _ in range(runs)]
                entry["profiler_kernel_us_median"] = {kk: statistics.median(x[kk] for x in per) for kk in KERNELS}
                entry["per_run"] = per
                res["p=%g r=%d R=%d" % (p, r, R)] = entry
            del pts, yx, values, outs
            torch.cuda.empty_cache()
    return res


def e2e(bgr, runs, steps):
    r, R, ratio = 4, 16, 0.64
    arms = {}
    for p in PERCENTS:
        pipe = LineEndPipeline(zoom_ratio=SCALE, peaks=p)
        rec, m = pipe.run_host_matches(bgr, r, R, ratio)
        arms["matches p=%g" % p] = ((lambda pipe: lambda: pipe.run_host_matches(bgr, r, R, ratio))(pipe),
                                    len(rec.points), int((m.next >= 0).sum()))
        arms["records p=%g" % p] = ((lambda pipe: lambda: pipe.run_host_records(bgr))(pipe), len(rec.points), None)
        arms["records_patch4 p=%g" % p] = ((lambda pipe: lambda: pipe.run_host_records(bgr, patch_radius=4))(pipe),
                                           len(rec.points), None)
    for fn, _, _ in arms.values():
        fn()
    ms = {k: [] for k in arms}
    for _ in range(runs):
        for k, (fn, _, _) in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
            ms[k].append((time.perf_counter() - t0) * 1000.0 / steps)
    return {k: {"points": pts, "matches": n, "ms_per_call": summary(ms[k])} for k, (_, pts, n) in arms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "matches_bench.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    record = {"card": card(), "runs": args.runs, "launches_per_run": LAUNCHES, "pan_dy_dx": PAN}
    host = torch.empty((64, 1080, 1920, 3), dtype=torch.uint8, pin_memory=True)
    host.numpy()[...] = panned_frames(4000, 64, 1080, 1920, PAN)
    bgr = host.numpy()
    frames = host.to(dev)
    record["matches"] = {"workload": "64 x 1080p BGR uint8 panned by %s per frame, scale sqrt2, 6 levels, 3 "
                                     "orientations, float32 outputs" % (PAN,), **matches(frames, args.runs)}
    del frames
    torch.cuda.empty_cache()
    record["e2e"] = {"workload": "run_host_matches(r=4, R=16, max_ratio=0.64) against run_host_records() and "
                                 "run_host_records(patch_radius=4), 64 x 1080p BGR uint8 page-locked, float32",
                     "steps_per_run": 3, **e2e(bgr, args.runs, 3)}
    record["card_after"] = card()
    with open(args.out, "w") as f:
        json.dump(record, f, indent=1)
    print(json.dumps(record["card"]))
    for k, v in record["matches"].items():
        if isinstance(v, dict):
            print("%s: %d points, %s, %s" % (k, v["points"], ", ".join(
                "ratio %s: %d matches, %.4f agree" % (rr[10:], v[rr]["matches"], v[rr]["agree_with_pan"])
                for rr in v if rr.startswith("max_ratio")), ", ".join(
                "%s %.2f us" % (a.replace("_kernel", ""), t) for a, t in v["profiler_kernel_us_median"].items())
                + ", call %.2f us (events)" % v["events_us_per_call"]["median"]))
    for arm, v in record["e2e"].items():
        if isinstance(v, dict):
            m = v["ms_per_call"]
            print("e2e %s: %d points, %.3f ms [%.3f-%.3f]" % (arm, v["points"], m["median"], m["min"], m["max"]))


if __name__ == "__main__":
    main()
