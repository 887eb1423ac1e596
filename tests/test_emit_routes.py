"""Every route of the feature-point emit, and the points-capacity contract, against the plain reference.

The emit (``csrc/emit.cu``) picks one of six routes by level shape, by batch and by the data:

R1  3-orientation pipeline, region edges on multiples of 8 columns, <= 1024 stack_b tiles and <= 2048 rows per level,
    every level <= 64 hits: stack_b reduces the window maxima, emit_count_kernel hands each level's sorted hits to
    emit_write_kernel.
R2  as R1, but some level has > 64 hits: emit_write_kernel walks the rows and the candidate tiles (beyond 32 tile
    columns it re-tests the tiles instead of reading its ballot).
R3  3-orientation pipeline, region edges off multiples of 8: window_max_kernel, then emit_count / emit_write.
R4  3-orientation pipeline, > 1024 tiles or > 2048 rows: the row kernels on stack_b's window maxima.
R5  fused orientation banks: window_max_kernel, then the row kernels.
R6  the stand-alone ``silent_max_value_indices_region``: window_max_kernel over row slices, then the row kernels.

The reference is ``oracle.silent_oracle.max_value_indices_region`` (max-pool, nearest upsample, ``>=``, argwhere) on the
bit-defined gray of the C oracle; the C oracle's own emit must give the same rows. The CPU test below proves that each
case exercises the route and the property it is listed for; the GPU tests check the rows, the profiler's kernel names
and the capacity contract (the first ``min(capacity, total)`` rows, ``count == total``, nothing written past
``capacity``).
"""
import ctypes
import functools
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, structured_frame, synthetic_frame

SQRT2 = 2 ** .5
SENTINEL = -0x5EE7
EMIT_MAX_TILES, EMIT_MAX_ROWS, EMIT_COMPACT = 1024, 2048, 64


# ---- mirror of the route choice (emit.cu: pool_geometry, window_geometry, max_value_indices_region; stack_fused.cu:
# ---- stack_tile_grid / pick_tile_w) ------------------------------------------------------------------------------------

def pool_geometry(h, w, rh, rw):
    """(oh, ow, pad top, pad left) of the SAME max-pool whose window is the whole level and whose stride is the region."""
    oh, ow = -(-h // rh), -(-w // rw)
    return oh, ow, max((oh - 1) * rh, 0) // 2, max((ow - 1) * rw, 0) // 2


def windows_fused(h, w, rh, rw):
    """Whether stack_b reduces the window maxima: <= 2 x 2 windows whose column edges sit on multiples of 8."""
    oh, ow, _, pl = pool_geometry(h, w, rh, rw)
    if oh > 2 or ow > 2:
        return False
    for j in range(ow):
        x0, x1 = max(j * rw - pl, 0), min(j * rw - pl + w, w)
        if x0 % 8 or (x1 % 8 and x1 != w):
            return False
    return True


def tile_grid(h, w):
    """stack_b's tiles: 16 rows by 48 or 64 columns, whichever wastes fewer columns of the last tile (64 on a tie)."""
    tw = 48 if -(-w // 48) * 48 < -(-w // 64) * 64 else 64
    return 16, tw, -(-h // 16), -(-w // tw)


def predict_route(h, w, bank, level_hits, standalone=False):
    if standalone:
        return "R6"
    if bank:
        return "R5"
    _, _, nty, ntx = tile_grid(h, w)
    if nty * ntx > EMIT_MAX_TILES or h > EMIT_MAX_ROWS:
        return "R4"
    if not windows_fused(h, w, h // 2, w // 2):
        return "R3"
    return "R2" if max(level_hits, default=0) > EMIT_COMPACT else "R1"


def predict_kernels(route, h, w):
    """Emit kernels that run (True) and that must not run (False) on a route."""
    one_cta = route in ("R1", "R2", "R3")
    fused = route in ("R1", "R2", "R4") and windows_fused(h, w, h // 2, w // 2)
    return {"window_max_kernel": not fused, "emit_count_kernel": one_cta, "emit_write_kernel": one_cta,
            "count_rows_kernel": not one_cta, "scan_level_kernel": not one_cta, "write_rows_kernel": not one_cta}


def capacity_boundaries(pts):
    """Capacities to truncate at: 0, 1, total - 1, total, one inside a row's run of hits (row cap - 1 and row cap share
    level and y) and one at a level boundary (row cap is the first of its level). None for a missing kind."""
    total = len(pts)
    same_row = np.nonzero((pts[1:, :2] == pts[:-1, :2]).all(axis=1))[0] + 1
    level_edge = np.nonzero(pts[1:, 0] != pts[:-1, 0])[0] + 1
    mid_run = int(same_row[len(same_row) // 2]) if len(same_row) else None
    edge = int(level_edge[len(level_edge) // 2]) if len(level_edge) else None
    return dict(zero=0, one=1, total_minus_1=total - 1, total=total, in_row=mid_run, level_edge=edge)


# ---- cases ---------------------------------------------------------------------------------------------------------------

def periodic_frame(p, seed, h, w):
    """A random p x p tile repeated: level 0 (crop = output size, sampled at integer positions) gets a periodic gray,
    so each window's maximum is reached many times, bit for bit."""
    tile = np.random.RandomState(seed).randint(0, 256, size=(p, p, 3)).astype(np.uint8)
    return np.ascontiguousarray(np.tile(tile, (h // p + 1, w // p + 1, 1))[:h, :w])


def _frame(spec, h, w):
    kind = spec[0]
    if kind == "noise":
        return synthetic_frame(spec[1], spec[2], h, w)
    if kind == "struct":
        return structured_frame(spec[1], h, w)
    return periodic_frame(spec[1], spec[2], h, w)


# name: frames (specs), frame (H, W), output_size (w, h), zoom, orientations, route, extra property
# "wide": a level > 64 hits with hits in tile columns >= 32; "order": > 256 levels in one call; "trunc": the capacity
# contract runs on this case
PIPE_CASES = {
    "r1_noise_288x192": ([("noise", 11, i) for i in range(3)], (480, 640), (288, 192), 1.3, None, "R1", ()),
    # (the structured frames' black patch makes every window of their levels NaN: levels without hits in between)
    "r1_struct_96x64": ([("struct", 21), ("noise", 21, 0), ("struct", 22)], (240, 320), (96, 64), 1.5, None, "R1", ()),
    "r1_periodic_96x64": ([("periodic", 12, 1), ("noise", 12, 0), ("struct", 3)], (480, 640), (96, 64), 1.3, None,
                          "R1", ("trunc",)),
    "r3_72x48": ([("periodic", 4, 1), ("noise", 13, 0), ("struct", 3)], (240, 320), (72, 48), 1.5, None, "R3",
                 ("trunc",)),
    "r3_100x66": ([("struct", 31), ("noise", 14, 0), ("struct", 32)], (300, 400), (100, 66), 1.4, None, "R3", ()),
    "r2_periodic_96x64": ([("periodic", 4, 1), ("noise", 15, 0), ("struct", 4)], (480, 640), (96, 64), 1.3, None,
                          "R2", ("trunc",)),
    "r2_wide_1632x96": ([("periodic", 8, 2), ("noise", 9, 0)], (1080, 1920), (1632, 96), SQRT2, None, "R2",
                        ("wide", "trunc")),
    "r4_wide_2112x512": ([("noise", 5, 0), ("periodic", 8, 3)], (2160, 3840), (2112, 512), math.e ** .5, None, "R4",
                         ("trunc",)),
    "r4_tall_64x2112": ([("noise", 5, 0), ("periodic", 8, 3)], (2400, 100), (64, 2112), 1.5, None, "R4", ("trunc",)),
    "order_r1_48x": ([("noise", 16, i) for i in range(48)], (480, 640), (96, 64), 1.3, None, "R1", ("order",)),
    "order_r5_48x": ([("noise", 17, i) for i in range(48)], (480, 640), (96, 64), 1.3, 4, "R5", ("order",)),
}
for _nb in (4, 8, 12, 16):   # the fused banks at w % 4 != 0 and w % 4 == 0 (bank frames: 16-byte BGR rows)
    PIPE_CASES["r5_b%d_34x18" % _nb] = ([("periodic", 4, _nb), ("noise", 18, _nb), ("struct", _nb)], (48, 64), (34, 18),
                                        SQRT2, _nb, "R5", ("trunc",) if _nb == 8 else ())
    PIPE_CASES["r5_b%d_48x32" % _nb] = ([("periodic", 4, _nb), ("noise", 19, _nb), ("struct", _nb)], (96, 128), (48, 32),
                                        SQRT2, _nb, "R5", ())
PIPE_ENTRIES = {name: ("device", "host") if c[4] is None and not name.startswith("order") else ("device",)
                for name, c in PIPE_CASES.items()}


def _standalone_values():
    """R6 cases: name -> (value [n, h, w, 1] float32, region_h, region_w)."""
    rs = np.random.RandomState(606)
    cases = {}
    v = np.round(rs.randn(3, 130, 67) * 4).astype(np.float32) / 4 - 6    # negative, with ties
    cases["negative_w67"] = (v, 65, 34)
    v = np.full((2, 160, 40), -1.0, np.float32)                            # +0 / -0 in different row slices of a window
    v[0, 3, 5], v[0, 150, 30] = -0.0, 0.0
    v[1, 2::40, 7], v[1, 155, 1::9] = 0.0, -0.0
    cases["signed_zero_w40"] = (v, 80, 20)
    v = rs.randn(2, 128, 52).astype(np.float32)
    v[0] = -np.inf                                                         # an all -inf level
    v[1, 100:, :26] = -np.inf
    cases["neg_inf_w52"] = (v, 64, 26)
    v = np.round(rs.rand(2, 144, 44) * 8).astype(np.float32)
    v[0, 77, 40] = np.nan                                                  # NaN in exactly one row slice
    cases["nan_one_slice_w44"] = (v, 72, 22)
    cases["all_equal_w50"] = (np.full((2, 40, 50), 3.5, np.float32), 20, 25)
    cases["region_not_dividing_w70"] = (np.round(rs.rand(2, 50, 70) * 6).astype(np.float32), 15, 22)
    cases["region_larger_w30"] = (rs.rand(2, 20, 30).astype(np.float32), 25, 40)
    cases["region_1x1_w36"] = (np.round(rs.rand(1, 24, 36) * 3).astype(np.float32), 1, 1)
    cases["regions_4096_w64"] = (np.round(rs.rand(1, 64, 64) * 3).astype(np.float32), 1, 1)
    cases["levels_300_w12"] = (np.round(rs.rand(300, 8, 12) * 2).astype(np.float32), 4, 6)
    cases["ties_w52"] = (np.round(rs.rand(3, 40, 52) * 2).astype(np.float32), 20, 26)
    return {k: (np.ascontiguousarray(v[..., None]), rh, rw) for k, (v, rh, rw) in cases.items()}


STANDALONE_CASES = _standalone_values()
STANDALONE_TRUNC = ("ties_w52", "levels_300_w12")


def case_frames(name):
    specs, (H, W) = PIPE_CASES[name][:2]
    return np.stack([_frame(s, H, W) for s in specs])


@functools.lru_cache(maxsize=None)
def pipe_reference(name):
    """frames, pyramid and the C oracle's stack of a pipeline case, plus the literal reference points."""
    from oracle import c_oracle, silent_oracle as lit
    from pysilent_b200.pipeline import orientation_bank_filters
    import pysilent_b200.constant_convolutions as cc
    _, _, size, zoom, nb, _, _ = PIPE_CASES[name]
    frames = case_frames(name)
    pyr = c_oracle.from_image(frames, 3, size, zoom)
    n, h, w = pyr.shape[:3]
    if nb is None:
        f = dict(rgc=cc.midget_rgc(2), rgby=cc.rgby_3(2), stripe=cc.rgb_2d_stripe_tensors(),
                 blur=cc.blur_tensor(2, lengths=7), end=cc.rgb_2d_end_tensors())
        ref = c_oracle.line_end_stack(pyr, f)
    else:
        ref = c_oracle.bank_stack(pyr, orientation_bank_filters(nb), (h // 2, w // 2))
    pts = lit.max_value_indices_region(ref["gray"], [1, h // 2, w // 2, 1], ref["gray"])
    return dict(frames=frames, n=n, h=h, w=w, orient=ref["orient"], padded=ref["padded"], gray=ref["gray"], points=pts,
                c_points=ref["points"], hits=np.bincount(pts[:, 0], minlength=n))


@functools.lru_cache(maxsize=None)
def standalone_reference(name):
    from oracle import silent_oracle as lit
    v, rh, rw = STANDALONE_CASES[name]
    return lit.max_value_indices_region(v, [1, rh, rw, 1], v)


# ---- CPU: the case list proves its routes --------------------------------------------------------------------------------

def test_route_mirror_matches_the_kernel_limits():
    assert tile_grid(192, 288)[1:] == (48, 12, 6) and tile_grid(512, 2112)[1:] == (64, 32, 33)
    assert tile_grid(96, 1632)[1:] == (48, 6, 34) and tile_grid(2112, 64)[1:] == (64, 132, 1)
    assert windows_fused(192, 288, 96, 144) and windows_fused(64, 96, 32, 48) and windows_fused(512, 2112, 256, 1056)
    assert not windows_fused(48, 72, 24, 36) and not windows_fused(66, 100, 33, 50)
    assert pool_geometry(64, 64, 1, 1)[:2] == (64, 64) and pool_geometry(17, 241, 1, 1)[:2] == (17, 241)


def test_cases_cover_every_route_and_property(c_oracle):
    covered = set()
    for name, (_, _, size, _, nb, route, props) in PIPE_CASES.items():
        ref = pipe_reference(name)
        h, w, hits = ref["h"], ref["w"], ref["hits"]
        assert (h, w) == (size[1], size[0]), name
        assert np.array_equal(ref["points"], ref["c_points"]), name + ": the two oracles disagree"
        got = predict_route(h, w, nb is not None, hits)
        assert got == route, "%s: predicted %s, listed as %s (hits per level %s)" % (name, got, route, hits)
        covered.add(route)
        _, tw, nty, ntx = tile_grid(h, w)
        if route == "R1":
            assert hits.max() <= EMIT_COMPACT and hits.sum() > 0, name
        if route == "R2":
            assert hits.max() > EMIT_COMPACT, name
        if route == "R4":
            assert nty * ntx > EMIT_MAX_TILES or h > EMIT_MAX_ROWS, name
            assert hits.max() > EMIT_COMPACT and (hits[hits > 0] <= 4).any(), name + ": a few-hit and a many-hit level"
        if "wide" in props:
            many = np.nonzero(hits > EMIT_COMPACT)[0]
            pts = ref["points"]
            assert ntx > 32 and (pts[np.isin(pts[:, 0], many), 2] // tw >= 32).any(), name
            covered.add("ntx>32")
        if "order" in props:
            assert ref["n"] > 256, name
            covered.add("order " + route)
        if "trunc" in props:
            caps = capacity_boundaries(ref["points"])
            assert caps["in_row"] is not None and caps["level_edge"] is not None, name
            assert 1 < caps["in_row"] < len(ref["points"]) - 1 and 1 < caps["level_edge"] < len(ref["points"]) - 1, caps
            covered.update("trunc %s %s" % (route, k) for k in caps)
    w_mod4 = set()
    for name, (v, rh, rw) in STANDALONE_CASES.items():
        pts = standalone_reference(name)
        c_pts, count = c_oracle.max_value_indices_region(v, (rh, rw))
        assert count == len(pts) and np.array_equal(pts, c_pts), name + ": the two oracles disagree"
        n, h, w = v.shape[:3]
        assert predict_route(h, w, False, [], standalone=True) == "R6"
        oh, ow = pool_geometry(h, w, rh, rw)[:2]
        assert oh * ow <= 4096, name
        w_mod4.add(w % 4 == 0)
        if name in STANDALONE_TRUNC:
            caps = capacity_boundaries(pts)
            assert caps["in_row"] is not None and caps["level_edge"] is not None, name
            covered.update("trunc R6 %s" % k for k in caps)
    covered.add("R6")
    assert w_mod4 == {True, False}
    assert pool_geometry(*STANDALONE_CASES["regions_4096_w64"][0].shape[1:3], 1, 1)[:2] == (64, 64)
    # the row-slice cases: 16 slices (h >= 128), the -0 / +0 pair and the NaN in different slices of one window
    assert all(STANDALONE_CASES[k][0].shape[1] >= 128 for k in ("signed_zero_w40", "neg_inf_w52", "nan_one_slice_w44"))
    want = {"R1", "R2", "R3", "R4", "R5", "R6", "ntx>32", "order R1", "order R5"}
    want |= {"trunc %s %s" % (r, k) for r in ("R1", "R2", "R3", "R4", "R5", "R6")
             for k in ("zero", "one", "total_minus_1", "total", "in_row", "level_edge")}
    assert want <= covered, sorted(want - covered)


# ---- GPU -----------------------------------------------------------------------------------------------------------------

def _torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def cuda(built_lib):
    torch = _torch()
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert built_lib.silent_device_count() >= 1
    return torch


def _pipe(name):
    from pysilent_b200 import LineEndPipeline
    _, _, size, zoom, nb, _, _ = PIPE_CASES[name]
    return LineEndPipeline(output_size=size, zoom_ratio=zoom, orientations=nb)


def _assert_bits(got, want, what):
    got = got.detach().cpu().numpy() if hasattr(got, "detach") else np.asarray(got)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    same = (got == want) | (np.isnan(got) & np.isnan(want))
    assert same.all() and np.array_equal(np.isnan(got), np.isnan(want)), \
        "%s: %d of %d values differ from the C oracle" % (what, (~same).sum(), same.size)


def _kernels_run(torch, fn):
    """Names of the CUDA kernels ``fn`` launched, from torch.profiler."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.name for e in prof.events() if e.device_type == DeviceType.CUDA})


def witness_all():
    """Kernel names of one call per case: ``{pipeline case: names, "standalone " + case: names}``. Each pipeline is run
    once before its recorded call, so that plan set-up stays out of the record."""
    import torch
    from pysilent_b200 import _ops
    seen = {}
    for name in sorted(PIPE_CASES):
        pipe = _pipe(name)
        frames = torch.from_numpy(case_frames(name)).cuda()
        pipe.run_frames(frames)
        seen[name] = _kernels_run(torch, lambda: pipe.run_frames(frames))
    for name, (v, rh, rw) in sorted(STANDALONE_CASES.items()):
        dv = torch.from_numpy(v).cuda()
        seen["standalone " + name] = _kernels_run(torch, lambda: _ops.max_value_indices_region(dv, rh, rw))
    return seen


_WITNESS_SCRIPT = """
import json, sys
sys.path[:0] = [%r, %r]
import test_emit_routes
print("ROUTES " + json.dumps(test_emit_routes.witness_all()))
"""


@pytest.fixture(scope="module")
def route_witness(cuda):
    """The profiler's record of every case, taken in a child process: the profiler sessions stay out of the test
    process, whose later sessions (other tests record kernel names too) then start from a profiler never used there."""
    tests = os.path.dirname(os.path.abspath(__file__))
    flags = ["-s"] if sys.flags.no_user_site else []
    run = subprocess.run([sys.executable] + flags + ["-c", _WITNESS_SCRIPT % (tests, ROOT)], cwd=ROOT,
                         capture_output=True, text=True, timeout=900)
    lines = [line for line in run.stdout.splitlines() if line.startswith("ROUTES ")]
    assert run.returncode == 0 and lines, "route witness failed (%d):\n%s" % (run.returncode, run.stderr[-4000:])
    return json.loads(lines[-1][len("ROUTES "):])


def _assert_route(names, route, h, w, what):
    assert names, "%s: the profiler reported no CUDA events" % what
    for kernel, expected in predict_kernels(route, h, w).items():
        ran = any(kernel in n for n in names)
        assert ran == expected, "%s (%s): %s %s, kernels seen: %s" % (
            what, route, kernel, "did not run" if expected else "ran", names)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PIPE_CASES))
def test_pipeline_points_against_reference(name, cuda, route_witness):
    torch = cuda
    ref = pipe_reference(name)
    pipe = _pipe(name)
    frames = torch.from_numpy(ref["frames"]).cuda()
    _assert_route(route_witness[name], PIPE_CASES[name][5], ref["h"], ref["w"], name)
    res = pipe.run_frames(frames)
    _assert_bits(res.orient, ref["orient"], name + " orient")
    _assert_bits(res.padded_line_end, ref["padded"], name + " padded_line_end")
    pts = res.points.cpu().numpy()
    assert pts.dtype == np.int64 and np.array_equal(pts, ref["points"]), "%s points: %d rows, reference %d" % (
        name, len(pts), len(ref["points"]))
    if "host" in PIPE_ENTRIES[name]:
        host = pipe.run_host(ref["frames"])
        _assert_bits(host.orient, ref["orient"], name + " host orient")
        _assert_bits(host.padded_line_end, ref["padded"], name + " host padded_line_end")
        assert np.array_equal(host.points, ref["points"]), name + " host points"


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(n for n, c in PIPE_CASES.items() if "order" in c[6]))
def test_points_of_a_batch_are_the_per_frame_points_in_order(name, cuda):
    """More than 256 levels in one call: the whole points array is the concatenation of every frame's own points,
    level ids offset by the levels of the frames before (the level totals are summed in several rounds)."""
    torch = cuda
    ref = pipe_reference(name)
    L = ref["n"] // len(ref["frames"])
    parts = []
    for i in range(len(ref["frames"])):
        own = ref["points"][(ref["points"][:, 0] >= i * L) & (ref["points"][:, 0] < (i + 1) * L)]
        parts.append(own)
    want = np.concatenate(parts)
    got = _pipe(name).run_frames(torch.from_numpy(ref["frames"]).cuda()).points.cpu().numpy()
    assert len(want) == len(ref["points"]) and np.array_equal(got, want)
    assert np.all(np.diff(got[:, 0]) >= 0)


def _sentinel_points(torch, rows, device="cuda"):
    return torch.full((rows, 4), SENTINEL, dtype=torch.int64, device=device)


def _check_truncated(big, cap, count, want, what):
    big = big.cpu().numpy() if hasattr(big, "cpu") else big
    k = min(cap, len(want))
    assert count == len(want), "%s cap %d: count %d, total %d" % (what, cap, count, len(want))
    assert np.array_equal(big[:k], want[:k]), "%s cap %d: the first %d rows differ" % (what, cap, k)
    assert (big[cap:] == SENTINEL).all(), "%s cap %d: rows past the capacity were written" % (what, cap)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(n for n, c in PIPE_CASES.items() if "trunc" in c[6]))
def test_pipeline_capacity_contract(name, cuda):
    """run_frames(out=...) and silent_pipeline_run_host with a points buffer of ``cap`` rows inside a larger one."""
    torch = cuda
    from pysilent_b200 import _lib, _ops
    ref = pipe_reference(name)
    want = ref["points"]
    pipe = _pipe(name)
    nb = PIPE_CASES[name][4]
    frames = torch.from_numpy(ref["frames"]).cuda()
    orient = torch.empty((ref["n"], ref["h"], ref["w"], nb or 3), dtype=torch.float32, device="cuda")
    line_end = torch.empty_like(orient)
    host_orient = np.empty(tuple(orient.shape), np.float32)
    host_line_end = np.empty_like(host_orient)
    for kind, cap in capacity_boundaries(want).items():
        big = _sentinel_points(torch, len(want) + 64)
        count = torch.full((1,), -1, dtype=torch.int64, device="cuda")
        pipe.run_frames(frames, out=(orient, line_end, big[:cap], count))
        torch.cuda.synchronize()
        _check_truncated(big, cap, int(count.item()), want, "%s device %s" % (name, kind))
        if "host" not in PIPE_ENTRIES[name]:
            continue
        plan = pipe.plan_for(frames)
        host = np.full((len(want) + 64, 4), SENTINEL, np.int64)
        hcount = ctypes.c_int64(-1)
        with torch.cuda.device(frames.device):
            _lib.check(_lib.lib().silent_pipeline_run_host(
                plan.handle, ctypes.byref(pipe.stack_weights()), ref["frames"].ctypes.data, len(ref["frames"]),
                host_orient.ctypes.data, host_line_end.ctypes.data, host.ctypes.data, cap, ctypes.byref(hcount),
                _ops.stream_ptr()), "silent_pipeline_run_host")
        _check_truncated(host, cap, hcount.value, want, "%s host %s" % (name, kind))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(STANDALONE_CASES))
def test_standalone_points_against_reference(name, cuda, route_witness):
    torch = cuda
    from pysilent_b200 import _ops
    from pysilent_b200.util.selection import max_value_indices_region
    v, rh, rw = STANDALONE_CASES[name]
    want = standalone_reference(name)
    dv = torch.from_numpy(v).cuda()
    _assert_route(route_witness["standalone " + name], "R6", v.shape[1], v.shape[2], name)
    got = _ops.max_value_indices_region(dv, rh, rw).cpu().numpy()
    assert np.array_equal(got, want), "%s: %d rows, reference %d" % (name, len(got), len(want))
    via_util = max_value_indices_region(dv, [1, rh, rw, 1], dv).cpu().numpy()
    assert np.array_equal(via_util, want), name + " (util.selection)"
    # the same values at an address that is 4 but not 16 bytes aligned (a contiguous view at an odd offset)
    flat = torch.empty(v.size + 1, dtype=torch.float32, device="cuda")
    shifted = flat[1:].view(v.shape)
    shifted.copy_(dv)
    assert shifted.data_ptr() % 16 != 0
    assert np.array_equal(_ops.max_value_indices_region(shifted, rh, rw).cpu().numpy(), want), name + " (unaligned)"


@pytest.mark.gpu
def test_standalone_region_count_limit(cuda):
    torch = cuda
    from pysilent_b200 import _ops
    ok = torch.from_numpy(STANDALONE_CASES["regions_4096_w64"][0]).cuda()
    assert np.array_equal(_ops.max_value_indices_region(ok, 1, 1).cpu().numpy(),
                          standalone_reference("regions_4096_w64"))
    too_many = torch.zeros((1, 17, 241, 1), dtype=torch.float32, device="cuda")   # 17 x 241 = 4097 regions
    with pytest.raises(RuntimeError, match=r"status -2\)"):
        _ops.max_value_indices_region(too_many, 1, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", STANDALONE_TRUNC)
def test_standalone_capacity_contract(name, cuda):
    torch = cuda
    from pysilent_b200 import _lib, _ops
    v, rh, rw = STANDALONE_CASES[name]
    want = standalone_reference(name)
    n, h, w = v.shape[:3]
    dv = torch.from_numpy(v).cuda()
    nbytes = _lib.lib().silent_selection_workspace_bytes(n, h, w)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    for kind, cap in capacity_boundaries(want).items():
        big = _sentinel_points(torch, len(want) + 64)
        count = torch.full((1,), -1, dtype=torch.int64, device="cuda")
        _lib.check(_lib.lib().silent_max_value_indices_region(
            _ops.ptr(dv), n, h, w, rh, rw, _ops.ptr(big), cap, _ops.ptr(count), _ops.ptr(ws), nbytes,
            _ops.stream_ptr()), "silent_max_value_indices_region")
        torch.cuda.synchronize()
        _check_truncated(big, cap, int(count.item()), want, "%s %s" % (name, kind))
        got = _ops.max_value_indices_region(dv, rh, rw, capacity=cap).cpu().numpy()
        assert np.array_equal(got, want[:cap]), "%s: _ops capacity %d" % (name, cap)
