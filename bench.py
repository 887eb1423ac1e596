#!/usr/bin/env python
"""Benchmark of the slam_recognition filter-pipeline hot path on B200 (contract: see the driver's prompt / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]

A step = one pass of the hot path (pyramid -> S1-S7 fused stack -> feature-point emit) over one batch of synthetic
1080p uint8 BGR frames (BASELINE config C3: 1920x1080, scale sqrt(2) -> 6 levels of 192x288, batch 64 per GPU; frames of
a video batch are independent, so N GPUs each process their own 64 frames: weak scaling, only the feature-point gather
crosses NVLink). Prints ONE JSON line on rank 0.

  value     frames/s, whole job, inputs resident in HBM, timed with CUDA events on the launching stream (max over ranks)
  e2e       same metric through LineEndPipeline.run_host (C-ABI silent_pipeline_run_host) with pinned HOST buffers:
            host->device copy of the frames and device->host copy of both result tensors + points inside the timed
            region; e2e.link relates it to a concurrent pinned H2D + D2H copy probe on the same ranks
  roofline  algorithmic bytes per step (SURVEY 8(d): union crop read once + the two output tensors) / device time of the
            step, against the measured HBM copy bandwidth in MEASURED_PEAKS.json
  configs   the other BASELINE configs (C1, C2, C4, C5) on this rank's GPU: frames/s, algorithmic bytes, roofline frac
  cpu_baseline  the reference's CPU path on the host cores: kind "port" (bit-defined C oracle, all cores) plus
            cpu_baseline.reference_python (scipy.ndimage.zoom pyramid exactly as from_image.py:55-59 calls it + the graph
            restated in numpy; real TensorFlow-1 cannot be installed here), for C1 and C3 frames
  ranks     per-rank device ms (min / median / max), host enqueue time per step, wait for the last point gather
  gather_check  (N > 1) rank 0 recomputes rank 1's frames locally and compares them with the rows NCCL delivered

--dump-outputs DIR writes what the last timed step handed its caller on rank 0 as DIR/<name>.npy (see dump_outputs), so
that two builds run with the same arguments (hence the same seeded frames) can be compared output for output.
"""
import argparse
import concurrent.futures
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the tree may be read-only and the bench writes nothing into it: no bytecode caches, in this process or its CPU workers
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

METRIC = "frames/sec (1080p RGB, full pyramid)"
CENTER = (288, 192)
# BASELINE.json configs, parametrised as in SURVEY 8(d): id -> (frame h, w), scale, levels, frames per GPU, orientations
CONFIGS = {
    1: dict(hw=(480, 640), scale=1.3, levels=4, batch=1, orient=None,
            name="C1: single 640x480 frame, 4-level pyramid (scale 1.3)"),
    2: dict(hw=(1080, 1920), scale=2 ** .5, levels=6, batch=1, orient=None,
            name="C2: one 1920x1080 frame per call, 6 levels"),
    3: dict(hw=(1080, 1920), scale=2 ** .5, levels=6, batch=64, orient=None,
            name="C3: 1080p video batch 64 per GPU, 6 levels"),
    4: dict(hw=(2160, 3840), scale=2 ** .5, levels=8, batch=16, orient=8,
            name="C4: 3840x2160, 8 levels, 8-orientation bank, batch 16"),
    5: dict(hw=(720, 1280), scale=2 ** .5, levels=5, batch=32, orient=None,
            name="C5: 1280x720 camera streams, 5 levels, 32 streams per GPU (256 on 8 GPUs) + NCCL point gather"),
}
HEADLINE = 3
WORKLOAD = ("C3: 1920x1080 uint8 BGR frames, scale sqrt2 -> 6 levels of 192x288x3, full stack (pyramid + center-surround + "
            "stripe/regulator + line-end + feature points), batch %d per GPU")


def synthetic_frames(config, first, count):
    """uint8 uniform noise, RandomState(1000 * config + global_frame_index) (SURVEY 8(d))."""
    hw = CONFIGS[config]["hw"]
    out = np.empty((count,) + hw + (3,), np.uint8)
    for i in range(count):
        out[i] = np.random.RandomState(1000 * config + first + i).randint(0, 256, size=hw + (3,))
    return out


def default_filters():
    import pysilent_b200.constant_convolutions as cc
    return dict(rgc=cc.midget_rgc(2), rgby=cc.rgby_3(2), stripe=cc.rgb_2d_stripe_tensors(),
                blur=cc.blur_tensor(2, lengths=7), end=cc.rgb_2d_end_tensors())


# ---- CPU arms: the reference's path on the host cores -----------------------------------------------------------------

_WORKER = {}


def _cpu_worker_init(config, filters):
    """Worker process of the CPU arm: its own copy of the oracle library, two frames of the workload."""
    from oracle import c_oracle
    c_oracle.build()
    _WORKER.update(oracle=c_oracle, filters=filters, cfg=CONFIGS[config], frames=synthetic_frames(config, 0, 2))


def _cpu_worker_one(i):
    W = _WORKER
    pyr = W["oracle"].from_image(W["frames"][i % len(W["frames"])], 3, CENTER, W["cfg"]["scale"])
    return len(W["oracle"].line_end_stack(pyr, W["filters"])["points"])


class CpuPort:
    """The bit-defined C oracle (oracle/silent_oracle.c: pyramid + S1-S8, gcc -O3 -mavx2 -mfma), one frame per host core
    in flight: one worker PROCESS per core (spawned, numpy + the oracle library only -- threads of one process scale
    3x worse: their per-frame buffers are fresh mappings of one address space). One ROUND = `threads` frames."""

    def __init__(self, config=HEADLINE, threads=None):
        import multiprocessing
        from oracle import c_oracle
        c_oracle.build()
        self.oracle, self.filters = c_oracle, default_filters()
        self.cfg = CONFIGS[config]
        self.threads = threads or os.cpu_count() or 1
        self.frames = synthetic_frames(config, 0, 2)
        self.pool = concurrent.futures.ProcessPoolExecutor(
            self.threads, mp_context=multiprocessing.get_context("spawn"), initializer=_cpu_worker_init,
            initargs=(config, {k: np.asarray(v) for k, v in self.filters.items()}))

    def one(self, i):
        pyr = self.oracle.from_image(self.frames[i % len(self.frames)], 3, CENTER, self.cfg["scale"])
        return len(self.oracle.line_end_stack(pyr, self.filters)["points"])

    def round(self):
        return len(list(self.pool.map(_cpu_worker_one, range(self.threads))))

    def close(self):
        self.pool.shutdown(wait=True, cancel_futures=True)


def cpu_port_sample(budget_s, config=HEADLINE):
    port = CpuPort(config)
    port.one(0)
    t0 = time.perf_counter()
    port.one(0)
    single = time.perf_counter() - t0
    port.round()   # (untimed: the workers start up, build their tables)
    rounds = max(1, min(8, int(budget_s / max(single * 2.0, 1e-3))))
    t0 = time.perf_counter()
    done = sum(port.round() for _ in range(rounds))
    elapsed = time.perf_counter() - t0
    port.close()
    return dict(value=done / elapsed, unit="frames/s", cores=port.threads, kind="port",
                sample="%d frames of %s through oracle/silent_oracle.c (pyramid + S1-S8; gcc -O3 -mavx2 -mfma), %d worker "
                       "processes x %d rounds, %.1f s; single-frame latency %.3f s" % (done, port.cfg["name"], port.threads,
                                                                                      rounds, elapsed, single))


def reference_python_sample(config, repeats):
    """The reference's own CPU arithmetic, single-threaded as the reference runs it: scipy.ndimage.zoom per level and
    channel exactly as from_image.py:55-59 calls it, then the graph of recognition_testing.py:69-77,90-91 restated with
    numpy (float64 convolutions; TensorFlow 1.x is not installable in this image). Median of `repeats` after one
    warm-up (SURVEY 8(d))."""
    from oracle import silent_oracle as lit
    cfg, filters = CONFIGS[config], default_filters()
    frame = synthetic_frames(config, 0, 1)[0]
    pyr_s, stack_s = [], []
    for i in range(repeats + 1):
        t0 = time.perf_counter()
        pyr = lit.from_image_scipy(frame.astype(np.float32), 3, CENTER, cfg["scale"])
        t1 = time.perf_counter()
        lit.line_end_stack(pyr, filters)
        t2 = time.perf_counter()
        if i:
            pyr_s.append(t1 - t0)
            stack_s.append(t2 - t1)
    p, s = statistics.median(pyr_s), statistics.median(stack_s)
    return dict(value=1.0 / (p + s), unit="frames/s", cores=1, kind="reference-python", config=cfg["name"],
                pyramid_s=p, stack_s=s,
                sample="median of %d single frames: scipy.ndimage.zoom(order=5, prefilter=False) pyramid %.3f s + numpy "
                       "restatement of the S1-S8 graph %.3f s (real TF-1 unavailable)" % (repeats, p, s))


def run_reference(args, rank):
    """`--impl reference`: the reference's CPU path on this box's host cores. One STEP = one round of `threads` frames
    of the headline workload through the oracle port (all host cores); exactly --warmup + --steps rounds run."""
    if rank != 0:
        return
    port = CpuPort(HEADLINE)
    for _ in range(max(args.warmup, 1)):
        port.round()
    t0 = time.perf_counter()
    frames = sum(port.round() for _ in range(args.steps))
    elapsed = time.perf_counter() - t0
    port.close()
    fps = frames / elapsed
    base = dict(value=fps, unit="frames/s", cores=port.threads, kind="port",
                sample="%d steps x %d frames (one per host core, one worker process each) of the 1080p/L=6 workload "
                       "through oracle/silent_oracle.c (pyramid + S1-S8; gcc -O3 -mavx2 -mfma), %.1f s"
                       % (args.steps, port.threads, elapsed))
    if not args.no_cpu:
        base["reference_python"] = {"C1": reference_python_sample(1, 3), "C3": reference_python_sample(3, 2)}
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * elapsed / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD % args.batch, "frame": "1920x1080x3 uint8", "levels": 6,
                   "batch_per_gpu": args.batch,
                   "sample": "bounded sample of that workload: each step = %d frames (one per host core)" % port.threads},
        "cpu_baseline": base,
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference's CPU path restated (bit-defined oracle port, all host cores): TensorFlow 1.x is not "
                "installable, the reference itself cannot run; cpu_baseline.reference_python times scipy's zoom as the "
                "reference calls it",
    }
    print(json.dumps(line), file=RESULT_OUT, flush=True)


# ---- clocks ---------------------------------------------------------------------------------------------------------------

class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [l for (t, l) in self.lines if (t0 is None or t >= t0) and (t1 is None or t <= t1)] or \
               [l for (_, l) in self.lines]
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for row in rows:
            parts = [p.strip() for p in row.split(",")]
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- GPU arm ----------------------------------------------------------------------------------------------------------------

def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def ncu_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def time_device(fn, steps, warmup=3):
    """ms per call of fn() on the current stream (CUDA events, warm-up, synchronise on both sides)."""
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def config_entry(config, dev, peak, world, rank):
    """One of the other BASELINE configs on this GPU: device-resident frames, frames/s and roofline fraction."""
    import torch
    from pysilent_b200 import LineEndPipeline
    cfg = CONFIGS[config]
    B = cfg["batch"]
    frames = torch.from_numpy(synthetic_frames(config, rank * B, B)).to(dev)
    pipe = LineEndPipeline(zoom_ratio=cfg["scale"], orientations=cfg["orient"])
    if cfg["orient"] is None:
        plan = pipe.plan_for(frames)
        plan.reserve(B)
        n = B * plan.levels
        bufs = (torch.empty((n, plan.h, plan.w, 3), dtype=torch.float32, device=dev),
                torch.empty((n, plan.h, plan.w, 3), dtype=torch.float32, device=dev),
                torch.empty((64 * n, 4), dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev))
        levels, alg = plan.levels, plan.algorithmic_bytes
        fn = lambda: pipe.run_frames(frames, out=bufs)   # noqa: E731
    else:
        res = pipe.run_frames(frames[:1])
        levels = int(res.orient.shape[0])
        from pysilent_b200.util.zoom.from_image import PyramidPlan
        plan = PyramidPlan(frames.shape[1:], frames.dtype, 3, CENTER, cfg["scale"])
        crop = plan.algorithmic_bytes - 2 * levels * plan.h * plan.w * 3 * 4
        alg = crop + 2 * levels * plan.h * plan.w * cfg["orient"] * 4      # SURVEY 8(d): C = 8 for the two outputs
        fn = lambda: pipe.run_frames(frames, want_points=True)   # noqa: E731
    steps = 30 if B <= 2 else 6
    ms = time_device(fn, steps)
    fps = B / (ms * 1e-3)
    out = {"workload": cfg["name"], "frames_per_s_per_gpu": fps, "ms_per_step": ms, "batch": B, "levels": levels,
           "algorithmic_bytes_per_frame": int(alg), "achieved_gbs": alg * fps / 1e9, "frac": alg * fps / 1e9 / peak}
    del frames
    torch.cuda.empty_cache()
    return out


def link_probe(dev, world):
    """Concurrent pinned H2D + D2H copies on every rank at once (the e2e path's traffic pattern): GB/s per direction of
    THIS rank; with N ranks the host side is shared, which is what caps e2e at N > 1."""
    import torch
    import torch.distributed as dist
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
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        both()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / 4
    return {"h2d_and_d2h_concurrent_gbs_each": nbytes / dt / 1e9, "bytes_each_way": nbytes}


DUMP_SAMPLE = 1 << 22   # elements kept of each [B*L,h,w,3] result tensor: 16 MB of float32, 32 MB for the two
DUMP_LIMIT = 64 << 20   # bytes of one dump in all


def dump_outputs(out_dir, orient, padded_line_end, points, gathered=None):
    """Write the arrays the timed path handed its caller as ``out_dir/<name>.npy``: ``orient`` and ``padded_line_end``
    (float32; beyond DUMP_SAMPLE elements, the elements at the sorted unique flat indices of
    ``RandomState(0).randint(0, numel, DUMP_SAMPLE)``, which depend on the shape alone), ``points`` (the valid feature-point
    rows (level, y, x, 0), float64: exact for these integers) and, on several GPUs, ``gathered_points`` (every rank's rows
    as the point gather delivered them)."""
    import torch
    arrays = {}
    numel = orient.numel()
    if numel > DUMP_SAMPLE:
        index = np.unique(np.random.RandomState(0).randint(0, numel, size=DUMP_SAMPLE))
        index = torch.from_numpy(index).to(orient.device)
    for name, t in (("orient", orient), ("padded_line_end", padded_line_end)):
        arrays[name] = (t.reshape(-1)[index] if numel > DUMP_SAMPLE else t).cpu().numpy().astype(np.float32)
    arrays["points"] = points.cpu().numpy().astype(np.float64)
    if gathered is not None:
        arrays["gathered_points"] = gathered.cpu().numpy().astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, rank, local_rank, world):
    import ctypes
    import torch
    import torch.distributed as dist
    from pysilent_b200 import LineEndPipeline, _lib, distributed as sdist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_node = sdist.bind_to_device_numa_node(local_rank)   # page-locked buffers below land next to the GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = CONFIGS[HEADLINE]
    B = args.batch
    pipe = LineEndPipeline(zoom_ratio=cfg["scale"])
    host_frames = torch.empty((B,) + cfg["hw"] + (3,), dtype=torch.uint8).pin_memory()
    host_frames.numpy()[...] = synthetic_frames(HEADLINE, rank * B, B)
    frames = host_frames.to(dev, non_blocking=True)
    plan = pipe.plan_for(frames)
    L, h, w = plan.levels, plan.h, plan.w
    n = B * L
    cap = 64 * n
    bufs = (torch.empty((n, h, w, 3), dtype=torch.float32, device=dev), torch.empty((n, h, w, 3), dtype=torch.float32,
            device=dev), torch.empty((cap, 4), dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev))
    gather_cap = 8 * n   # rows per rank in the fixed-size all-gather (generic input: 1-4 points per level)
    # the path's only exchange: feature points to every rank over NCCL/NVLink, one all-gather per step on a side stream
    # (it overlaps the next step's kernels; the final barrier + synchronize below waits for the last one)
    gatherer = sdist.PointGather(gather_cap, L, dev, native=args.native_gather) if world > 1 else None

    def step():
        pipe.run_frames(frames, out=bufs)
        return gatherer.submit(bufs[2], bufs[3], rank * B) if gatherer is not None else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    # (started BEFORE the barrier: spawning nvidia-smi takes rank 0 about a millisecond, and a rank that enters the timed
    # region late holds every other rank up through the point gather -- the max over ranks then measures the skew)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    launches0 = _lib.lib().silent_launch_count()
    ev0, ev1, ev_k = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    t_wall0 = time.perf_counter()
    ev0.record()
    slot = None
    for _ in range(args.steps):
        slot = step()
    t_enqueued = time.perf_counter()
    ev_k.record()                      # the last step's kernels are done here ...
    if gatherer is not None and slot is not None:   # ... and its gather (side stream) belongs to the timed region too
        torch.cuda.current_stream().wait_event(gatherer.done[slot])
    ev1.record()
    barrier()
    t_wall1 = time.perf_counter()
    launches = _lib.lib().silent_launch_count() - launches0
    my_ms = ev0.elapsed_time(ev1) / args.steps
    ms = my_ms
    gather_wait_ms = ev_k.elapsed_time(ev1)
    enqueue_ms = (t_enqueued - t_wall0) * 1000.0 / args.steps
    count_points = int(bufs[3].item())

    # the rows NCCL delivered for rank 1's frames against a local recomputation of the same frames on rank 0
    gather_check = None
    if gatherer is not None:
        pts, counts = gatherer.result(slot)
        if rank == 0:
            other = torch.from_numpy(synthetic_frames(HEADLINE, 1 * B, B)).to(dev)
            ref = pipe.run_frames(other).points.clone()
            ref[:, 0] += 1 * n
            got = pts[(pts[:, 0] >= n) & (pts[:, 0] < 2 * n)]
            mine = pts[pts[:, 0] < n]
            ok = bool(torch.equal(got, ref)) and bool(torch.equal(mine, bufs[2][:count_points])) and \
                int(counts.sum().item()) == int(pts.shape[0]) and bool((pts[1:, 0] >= pts[:-1, 0]).all())
            gather_check = "ok" if ok else "MISMATCH"
            del other
    if args.dump_outputs and rank == 0:   # before the passes below run the step again into the same buffers
        dump_outputs(args.dump_outputs, bufs[0], bufs[1], bufs[2][:count_points],
                     pts if gatherer is not None else None)

    # per-stage device time (separate, untimed pass with the library's event hooks)
    _lib.check(_lib.lib().silent_plan_enable_timing(plan.handle, 1))
    stage = np.zeros((5, 5))
    for i in range(5):
        pipe.run_frames(frames, out=bufs)
        vals = [ctypes.c_float() for _ in range(5)]
        _lib.check(_lib.lib().silent_plan_stage_ms(plan.handle, *[ctypes.byref(v) for v in vals[:3]]))
        _lib.check(_lib.lib().silent_plan_stack_split_ms(plan.handle, ctypes.byref(vals[3]), ctypes.byref(vals[4])))
        stage[i] = [v.value for v in vals]
    _lib.check(_lib.lib().silent_plan_enable_timing(plan.handle, 0))
    stage_ms = stage[1:].mean(axis=0)   # pyramid, stack (a + b), emit, stack_a, stack_b

    # end to end through the host-buffer entry point
    orient_host = torch.empty((n, h, w, 3), dtype=torch.float32).pin_memory().numpy()
    line_end_host = torch.empty((n, h, w, 3), dtype=torch.float32).pin_memory().numpy()
    host_np = host_frames.numpy()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        res = pipe.run_host(host_np, orient_host, line_end_host)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        res = pipe.run_host(host_np, orient_host, line_end_host)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1000.0 / e2e_steps
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    probe = link_probe(dev, world)
    del orient_host, line_end_host

    rank_ms = [my_ms]
    if world > 1:
        t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = (float(v) for v in t.tolist())
        total_launches = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(total_launches)
        launches = int(total_launches.item())
        per_rank = torch.zeros((world, 4), dtype=torch.float64, device=dev)
        mine_row = torch.tensor([my_ms, enqueue_ms, gather_wait_ms, probe["h2d_and_d2h_concurrent_gbs_each"]],
                                dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(per_rank, mine_row)
        per_rank = per_rank.cpu().numpy()
        rank_ms = per_rank[:, 0].tolist()
        enqueue_all, wait_all, probe_all = per_rank[:, 1].tolist(), per_rank[:, 2].tolist(), per_rank[:, 3].tolist()
    else:
        enqueue_all, wait_all, probe_all = [enqueue_ms], [gather_wait_ms], [probe["h2d_and_d2h_concurrent_gbs_each"]]

    peak, peak_src = measured_peak()
    # the other BASELINE configs (C5 on every rank: its workload is per-GPU streams; the rest on rank 0 only)
    configs = {}
    if not args.no_configs:
        c5 = config_entry(5, dev, peak, world, rank)
        if world > 1:
            t = torch.tensor([c5["ms_per_step"]], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            c5["ms_per_step_max_over_ranks"] = float(t.item())
            c5["frames_per_s_all_gpus"] = world * c5["batch"] / (float(t.item()) * 1e-3)
        if rank == 0:
            configs["C5"] = c5
            for cid in (1, 2, 4):
                configs["C%d" % cid] = config_entry(cid, dev, peak, world, rank)
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    alg_bytes = plan.algorithmic_bytes            # per frame, SURVEY 8(d): 13,240,584 B at 1080p / L=6 / uint8
    achieved = alg_bytes * B / (ms * 1e-3) / 1e9
    traffic = ncu_traffic()
    fps = world * B / (ms * 1e-3)
    # per-kernel view (DESIGN.md section 4): each kernel's own algorithmic bytes per frame = what it must read + write
    level_bytes = L * h * w * 4
    crop_bytes = alg_bytes - 2 * 3 * level_bytes
    kernel_alg = {"pyramid_pair_kernel": crop_bytes + 3 * level_bytes,           # union crop in, planar pyramid out
                  "stack_a_kernel": 3 * level_bytes + level_bytes,               # pyramid in, channel-sum plane out
                  "stack_b_kernel": level_bytes + 2 * 3 * level_bytes + level_bytes}   # plane in; orient, line_end, gray out
    kernel_ms = {"pyramid_pair_kernel": stage_ms[0], "stack_a_kernel": stage_ms[3], "stack_b_kernel": stage_ms[4]}
    kernels = {}
    for name, kb in kernel_alg.items():
        gbs = kb * B / (kernel_ms[name] * 1e-3) / 1e9 if kernel_ms[name] > 0 else 0.0
        kernels[name] = {"ms": float(kernel_ms[name]), "algorithmic_bytes_per_launch": int(kb * B), "achieved": gbs,
                         "frac": gbs / peak, "share_of_step": float(kernel_ms[name] / max(stage_ms[:3].sum(), 1e-9)),
                         "traffic": (traffic or {}).get("kernels", {}).get(name)}
    dominant = max(kernel_ms, key=kernel_ms.get)
    h2d = B * cfg["hw"][0] * cfg["hw"][1] * 3
    d2h = 2 * n * h * w * 3 * 4 + 8 + 32 * len(res.points)
    e2e_gbs_each = max(h2d, d2h) / (e2e_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD % B, "frame": "1920x1080x3 uint8", "levels": L, "batch_per_gpu": B,
                   "parallelism": "frame-sharded dp%d, NCCL point gather" % world,
                   "l2": "inputs (%.0f MB) and outputs (%.0f MB) per step exceed the 126 MB L2; no flush needed" % (
                       h2d / 1e6, d2h / 1e6),
                   "points_per_step": count_points},
        "clocks": clocks,
        "e2e": {"value": world * B / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "numa_node_rank0": numa_node,
                "api": "LineEndPipeline.run_host -> silent_pipeline_run_host, pinned host buffers",
                "link": {"probe": "pinned H2D + D2H copies of 256 MiB each, concurrently, on all %d ranks at once" % world,
                         "probe_gbs_each_way_per_rank": probe_all, "probe_gbs_each_way_min": min(probe_all),
                         "e2e_gbs_larger_direction_per_rank": e2e_gbs_each,
                         "frac_of_probe": e2e_gbs_each / max(min(probe_all), 1e-9)}},
        "gpu_launches": int(launches),
        "ranks": {"device_ms_per_step": {"min": min(rank_ms), "median": statistics.median(rank_ms), "max": max(rank_ms),
                                         "all": rank_ms},
                  "host_enqueue_ms_per_step": {"max": max(enqueue_all), "all": enqueue_all},
                  "last_gather_wait_ms": {"max": max(wait_all), "all": wait_all},
                  "gather_rows_per_rank": gather_cap + 1 if world > 1 else 0,
                  "gather_api": ("silent_gather_points (ncclAllGather)" if args.native_gather else
                                 "torch.distributed.all_gather_into_tensor") if world > 1 else None},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic.get("dram_bytes_per_step") if traffic else None,
                     "kernel": "whole step per GPU: pyramid_pair_kernel + stack_a_kernel + stack_b_kernel (quick pass + "
                               "fix-up pass) + 2 emit kernels (the step's algorithmic bytes over the step's device time; "
                               "dominant kernel: %s)" % dominant,
                     "algorithmic_bytes_per_step": alg_bytes * B, "peak_source": peak_src,
                     "traffic_source": traffic.get("source") if traffic else None,
                     "stage_ms": {"pyramid": stage_ms[0], "stack_fused": stage_ms[1], "emit": stage_ms[2]},
                     "kernels": kernels},
        "configs": configs,
    }
    if gather_check is not None:
        line["gather_check"] = gather_check
    if args.natural:
        line["structured_input"] = structured_input_entry(pipe, dev, B, plan)
    if not args.no_cpu:
        base = cpu_port_sample(args.cpu_seconds)
        base["reference_python"] = {"C1": reference_python_sample(1, 5), "C3": reference_python_sample(3, 3)}
        base["C1_port"] = cpu_port_sample(3.0, 1)
        line["cpu_baseline"] = base
    print(json.dumps(line), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def structured_input_entry(pipe, dev, B, plan):
    """Secondary figure: the same step on frames with flat and black patches (tests/conftest.structured_frame), where
    the regulator's blur really falls below 1 and stack_b's fix-up pass has work to do."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import structured_frame
    few = np.stack([structured_frame(900 + i, 1080, 1920) for i in range(8)])
    frames = torch.from_numpy(np.concatenate([few] * (B // 8), axis=0)).to(dev)
    n = B * plan.levels
    bufs = (torch.empty((n, plan.h, plan.w, 3), dtype=torch.float32, device=dev),
            torch.empty((n, plan.h, plan.w, 3), dtype=torch.float32, device=dev),
            torch.empty((64 * n, 4), dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev))
    ms = time_device(lambda: pipe.run_frames(frames, out=bufs), 10)
    return {"workload": "C3 shape, frames with smooth / flat / black patches (NaN and gain paths active)",
            "ms_per_step": ms, "frames_per_s_per_gpu": B / (ms * 1e-3)}


RESULT_OUT = sys.stdout   # where the JSON line goes (main() saves the real stdout before redirecting fd 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64, help="frames per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C1/C2/C4/C5 entries")
    ap.add_argument("--no-natural", dest="natural", action="store_false")
    ap.add_argument("--native-gather", action="store_true",
                    help="point gather through silent_gather_points (ncclAllGather behind the C ABI) instead of torch's")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's results to DIR/<name>.npy (at most 64 MB, see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours: the CPU arm keeps only point counts")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries exactly ONE JSON line: file descriptor 1 is pointed at stderr for everything else that writes to it
    # (NCCL prints its version banner there from native code), the JSON line goes to the saved descriptor
    global RESULT_OUT
    sys.stdout.flush()
    RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
