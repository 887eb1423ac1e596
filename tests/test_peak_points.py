"""Peak feature points (``silent_peak_points``, ``silent_plan_peak_points``, ``LineEndPipeline(peaks=p)``).

Pixel (y, x) of a level v fires iff v > 0, v >= thr = float32(1 - p) * max(v) + float32(p) * min(v) (the threshold of
``top_value_points``) and v >= the NaN-propagating maximum of its 3 x 3 window (``max_pool_3x3``, SAME). The CPU tests
check the binding, every status code of the two C calls, the constructor's validation of ``peaks`` and the numpy
reference below against a brute-force loop. The GPU tests check the rows bit for bit against that reference on the
call's own gray, on every route of every entry point, and the capacity contract, the records and patches of peak
points, the host entry points and the kernels each call runs.
"""
import ctypes
import math
import os

import numpy as np
import pytest

from conftest import ROOT
from test_point_records import (CASES, SENTINEL, SQRT2, _bgr, _geometry_plan, _lib_status, _np, _pipe, _raw_plan,
                                random_nv12)
from pysilent_b200 import _lib

PEAK_KERNELS = ("level_threshold_kernel", "peak_count_kernel", "scan_level_kernel", "peak_base_kernel",
                "peak_write_kernel")
REGION_KERNELS = ("window_max_kernel", "count_rows_kernel", "write_rows_kernel", "emit_count_kernel",
                  "emit_write_kernel")
BAD_PEAKS = (True, False, np.bool_(True), "0.5", -0.1, 1.1, -1, 2, math.nan, math.inf, -math.inf, 0.5j, [0.5], (0.5,))


def peak_reference(value, p):
    """int64 rows (level, y, x, 0) of the peaks of ``value`` [n, h, w, 1] (or [n, h, w]), from the oracle's pieces: the
    float32 threshold of ``top_value_points`` and the NaN-propagating ``max_pool_3x3``."""
    from oracle import silent_oracle as so
    v = np.asarray(value, dtype=np.float32)
    if v.ndim == 3:
        v = v[..., None]
    mx = np.max(v, axis=(1, 2), keepdims=True)
    mn = np.float32(-1.0) * np.max(-v, axis=(1, 2), keepdims=True)
    with np.errstate(invalid="ignore"):   # (0 * inf = NaN: the threshold of a level holding an infinity at p = 0 or 1)
        thr = (np.float32(1.0 - p) * mx + np.float32(p) * mn).astype(np.float32)
        return np.argwhere((v > 0) & (v >= thr) & (v >= so.max_pool_3x3(v))).astype(np.int64)


def brute_force(value, p):
    """The rule written out pixel by pixel in Python floats rounded to float32 at each operation."""
    v = np.asarray(value, dtype=np.float32)
    n, h, w = v.shape[:3]
    f32 = lambda x: float(np.float32(x))  # noqa: E731
    rows = []
    for k in range(n):
        lvl = [[float(v[k, y, x].item()) for x in range(w)] for y in range(h)]
        flat = [a for r in lvl for a in r]
        if any(a != a for a in flat):
            continue   # thr is NaN: no comparison with it holds
        thr = f32(f32(f32(1.0 - p) * max(flat)) + f32(f32(p) * min(flat)))
        for y in range(h):
            for x in range(w):
                c = lvl[y][x]
                nbrs = [lvl[j][i] for j in range(max(y - 1, 0), min(y + 2, h)) for i in range(max(x - 1, 0), min(x + 2, w))]
                if c > 0 and c >= thr and all(c >= b for b in nbrs):
                    rows.append((k, y, x, 0))
    return np.array(rows, dtype=np.int64).reshape(-1, 4)


def small_values():
    rs = np.random.RandomState(5)
    cases = {
        "noise": rs.normal(size=(3, 7, 9)),
        "plateaus": np.round(rs.rand(3, 8, 11) * 2),
        "all_zero_and_noise": np.concatenate([np.zeros((1, 6, 5)), rs.rand(1, 6, 5)]),
        "one_row": rs.rand(2, 1, 13),
        "one_column": rs.rand(2, 13, 1),
        "one_pixel": np.array([[[2.0]], [[0.0]], [[-1.0]]]),
        "negative": -rs.rand(2, 5, 5),
        "flat": np.full((2, 4, 6), 3.0),
    }
    nan = rs.rand(2, 6, 7)
    nan[1, 3, 2] = np.nan
    cases["nan_level"] = nan
    inf = rs.rand(2, 5, 5)
    inf[0, 2, 2] = np.inf
    cases["inf"] = inf
    return {k: v.astype(np.float32) for k, v in cases.items()}


# ---- CPU -----------------------------------------------------------------------------------------------------------------

def test_symbols_exported_and_bound(built_lib):
    for name, nargs in (("silent_peak_points", 11), ("silent_plan_peak_points", 7)):
        assert name in _lib.SYMBOLS and hasattr(built_lib, name), name
        assert len(getattr(built_lib, name).argtypes) == nargs, name
    header = open(os.path.join(ROOT, "include", "silent_b200.h")).read()
    assert "int silent_peak_points(" in header and "int silent_plan_peak_points(" in header
    assert "#define SILENT_ABI_VERSION 1" in header and built_lib.silent_abi_version() == 1


def test_status_codes_before_any_cuda_call(built_lib):
    """Every check fails on the host: no call here reaches CUDA, with or without a device (fake device pointers; the
    plan is never reserved, so a plan call that passes every other check fails on the plan's gray)."""
    L = built_lib
    fake = ctypes.c_void_p(256)
    ws_bytes = L.silent_selection_workspace_bytes(4, 8, 8)
    good = dict(value=fake, n=4, h=8, w=8, p=0.5, points=fake, capacity=16, count=fake, ws=fake, ws_bytes=ws_bytes)

    def op(**kw):
        a = dict(good, **kw)
        return L.silent_peak_points(a["value"], a["n"], a["h"], a["w"], a["p"], a["points"], a["capacity"], a["count"],
                                    a["ws"], a["ws_bytes"], None)
    for kw in (dict(value=None), dict(count=None), dict(ws=None), dict(points=None), dict(n=0), dict(h=0), dict(w=0),
               dict(n=-1), dict(h=-5), dict(capacity=-1), dict(p=math.nan), dict(p=-0.01), dict(p=1.01),
               dict(p=math.inf), dict(p=-math.inf)):
        assert op(**kw) == _lib_status("INVAL"), kw
    assert b"silent_peak_points" in L.silent_last_error()
    for kw in (dict(n=65536, h=1, w=1, ws_bytes=1 << 40), dict(n=1, h=1 << 15, w=1 << 15, ws_bytes=1 << 40),
               dict(n=1, h=1 << 30, w=1, ws_bytes=1 << 40)):
        assert op(**kw) == _lib_status("SHAPE"), kw
    for kw in (dict(ws_bytes=ws_bytes - 1), dict(ws_bytes=0), dict(n=5, ws_bytes=ws_bytes),
               dict(capacity=0, points=None, ws_bytes=ws_bytes - 1), dict(p=0.0, ws_bytes=0), dict(p=1.0, ws_bytes=0),
               dict(p=-0.0, ws_bytes=0)):
        assert op(**kw) == _lib_status("CAPACITY"), kw
        assert b"workspace" in L.silent_last_error()

    plan = _raw_plan(L)
    zero = _raw_plan(L, H=64, W=96, center=(96, 64))   # frame no larger than the centre: 0 levels
    levels = L.silent_plan_levels(plan)
    assert levels > 0

    def on_plan(**kw):
        a = dict(plan=plan, batch=1, p=0.5, points=fake, capacity=16, count=fake)
        a.update(kw)
        return L.silent_plan_peak_points(a["plan"], a["batch"], a["p"], a["points"], a["capacity"], a["count"], None)
    try:
        for kw in (dict(plan=None), dict(count=None), dict(points=None), dict(batch=0), dict(batch=-2),
                   dict(capacity=-1), dict(p=math.nan), dict(p=-0.5), dict(p=1.5)):
            assert on_plan(**kw) == _lib_status("INVAL"), kw
        assert on_plan(plan=zero) == _lib_status("SHAPE")
        assert on_plan(batch=65535 // levels + 1) == _lib_status("SHAPE")
        for kw in ({}, dict(batch=65535 // levels), dict(capacity=0, points=None), dict(p=0.0), dict(p=1.0)):
            assert on_plan(**kw) == _lib_status("CAPACITY"), kw
            assert b"reserve" in L.silent_last_error()
    finally:
        L.silent_plan_destroy(plan)
        L.silent_plan_destroy(zero)


def test_constructor_validates_peaks():
    from pysilent_b200 import LineEndPipeline, _ops
    from pysilent_b200.recognition_testing import LineEndDisplayer
    for bad in BAD_PEAKS:
        with pytest.raises(ValueError, match="peaks"):
            LineEndPipeline(peaks=bad)
        with pytest.raises(ValueError, match="peaks"):
            _ops.peak_points(np.zeros((1, 4, 4, 1), np.float32), bad)
    for good, want in ((None, None), (0, 0.0), (1, 1.0), (0.5, 0.5), (np.float32(0.25), 0.25), (np.int64(1), 1.0),
                       (-0.0, 0.0)):
        assert LineEndPipeline(peaks=good).peaks == want
    assert LineEndPipeline().peaks is None
    assert LineEndDisplayer(output_size=(34, 18)).peaks is None


@pytest.mark.parametrize("p", (0.0, 0.1, 0.5, 0.9, 1.0))
@pytest.mark.parametrize("name", sorted(small_values()))
def test_reference_equals_brute_force(name, p):
    v = small_values()[name]
    got = peak_reference(v, p)
    assert np.array_equal(got, brute_force(v, p)), (name, p)
    if name == "nan_level":
        assert (got[:, 0] == 0).any() and not (got[:, 0] == 1).any()
    if name == "all_zero_and_noise":
        assert not (got[:, 0] == 0).any() and (got[:, 0] == 1).any()
    if name == "flat" and p == 1.0:
        assert len(got) == v.size   # a plateau fires on every pixel
    if name == "negative":
        assert len(got) == 0


# ---- GPU -----------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cuda(built_lib):
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def device_values():
    rs = np.random.RandomState(11)
    cases = {k: v[..., None] for k, v in small_values().items()}
    cases["random_192x288"] = rs.rand(6, 192, 288).astype(np.float32)[..., None]
    cases["plateaus_w_odd"] = np.round(rs.rand(5, 33, 101) * 3).astype(np.float32)[..., None]
    cases["w_6"] = np.round(rs.rand(7, 20, 6) * 2).astype(np.float32)[..., None]
    mixed = rs.rand(6, 64, 96).astype(np.float32)
    mixed[1] = 0
    mixed[2, 10, 17] = np.nan
    mixed[3, :, :] = np.round(mixed[3] * 2)
    mixed[4, :2] = 0
    mixed[4, :, -2:] = 0
    cases["zero_nan_plateau_levels"] = mixed[..., None]
    cases["levels_300_w12"] = rs.rand(300, 9, 12).astype(np.float32)[..., None]
    return cases


def _gpu_peaks(torch, v, p, offset=False, capacity=None):
    from pysilent_b200 import _ops
    if offset:   # the same values 4 bytes past a 16-byte boundary: the kernels take their scalar loads
        buf = torch.empty(v.size + 1, dtype=torch.float32, device="cuda")
        t = buf[1:].view(v.shape)
        t.copy_(torch.from_numpy(v))
        assert t.data_ptr() % 16 == 4 and t.is_contiguous()
    else:
        t = torch.from_numpy(v).cuda()
    return _np(_ops.peak_points(t, p, capacity))


@pytest.mark.gpu
@pytest.mark.parametrize("offset", (False, True), ids=("aligned", "offset4"))
@pytest.mark.parametrize("p", (0.0, 0.1, 0.5, 1.0))
@pytest.mark.parametrize("name", sorted(device_values()))
def test_standalone_rows_equal_the_reference(name, p, offset, cuda):
    v = device_values()[name]
    want = peak_reference(v, p)
    got = _gpu_peaks(cuda, v, p, offset)
    assert got.dtype == np.int64 and np.array_equal(got, want), (name, p, offset, len(got), len(want))


@pytest.mark.gpu
def test_standalone_dense_output(cuda):
    """Thousands of peaks per level with most rows holding some: integer plateaus at p = 1 (thr = min)."""
    v = np.round(np.random.RandomState(3).rand(32, 192, 288) * 2).astype(np.float32)[..., None]
    want = peak_reference(v, 1.0)
    assert len(want) > 32 * 5000 and len(np.unique(want[:, :2], axis=0)) > 0.9 * 32 * 192
    assert np.array_equal(_gpu_peaks(cuda, v, 1.0), want)


# name: case of test_point_records.CASES (frames, size, zoom, pipeline keywords, route)
ROUTE_CASES = ("f32_480p_b3", "f16_480p_b3", "struct_b3", "single_720p", "nv12_b3", "4k_b1_bank16", "pyramid_float_b8",
               "pyramid_w100_b12", "pyramid_w100_b8_f16", "convert_nv12_w100_b4", "bank4_b3", "bank8_b3", "bank12_b3",
               "bank16_b3", "bank8_f16_b1")


def _peak_pipe(torch, name, p, **extra):
    make, size, zoom, kw, route = CASES[name]
    kw = dict(kw, **extra)
    return _pipe(torch, size, zoom, dict(kw, peaks=p)), torch.from_numpy(make()).cuda(), route


def _f32_twin(torch, name, p):
    """The same case with float32 outputs: its padded_line_end gives the call's float32 gray."""
    make, size, zoom, kw, _ = CASES[name]
    kw = {k: v for k, v in kw.items() if k != "out_dtype"}
    return _pipe(torch, size, zoom, dict(kw, peaks=p))


def _call_gray(torch, res):
    from pysilent_b200 import _ops
    return _np(_ops.value_from_color(res.padded_line_end.float()))


@pytest.mark.gpu
@pytest.mark.parametrize("p", (0.1, 0.5, 1.0))
@pytest.mark.parametrize("name", ROUTE_CASES)
def test_run_frames_rows_equal_the_reference_on_the_calls_gray(name, p, cuda):
    torch = cuda
    from pysilent_b200.pipeline import CONVERT, PLAN, PYRAMID
    pipe, frames, route = _peak_pipe(torch, name, p)
    nv12 = pipe.frame_format == "nv12"
    batched = frames if frames.dim() == (3 if nv12 else 4) else frames.unsqueeze(0)
    assert pipe._frame_route(pipe.orientations, pipe.frame_format, batched.dtype, batched.shape) == \
        dict(plan=PLAN, pyramid=PYRAMID, convert=CONVERT)[route]
    twin = _f32_twin(torch, name, p)
    ref_res = twin.run_frames(frames)
    gray = _call_gray(torch, ref_res)
    want = peak_reference(gray, p)
    assert len(want) > 0, name
    assert np.array_equal(_np(ref_res.points), want), name
    if ref_res.gray is not None:
        assert np.array_equal(_np(ref_res.gray), gray, equal_nan=True), name
    res = pipe.run_frames(frames)
    assert np.array_equal(_np(res.points), want), name + ": outputs of %s" % pipe.out_dtype
    if pipe.out_dtype == torch.float16:   # the float32 call's points and outputs rounded once
        assert np.array_equal(_np(res.orient), _np(ref_res.orient.half()), equal_nan=True)
    region = _pipe(torch, *CASES[name][1:4]).run_frames(frames)   # peaks change the points only
    assert np.array_equal(_np(region.orient.float()), _np(res.orient.float()), equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ("struct_b3", "bank8_b3", "bank16_b3"))
def test_call_gray_equals_the_c_oracle(name, c_oracle, cuda):
    """On small frames the gray the reference reads is the C oracle's gray, bit for bit."""
    torch = cuda
    from pysilent_b200.pipeline import orientation_bank_filters
    make, size, zoom, kw, _ = CASES[name]
    pipe = _pipe(torch, size, zoom, dict(kw, peaks=0.5))
    frames = make()
    res = pipe.run_frames(torch.from_numpy(frames).cuda())
    pyr = c_oracle.from_image(frames, 3, size, zoom)
    h, w = pyr.shape[1:3]
    if pipe.orientations is None:
        ref = c_oracle.line_end_stack(pyr, pipe.filters())
    else:
        ref = c_oracle.bank_stack(pyr, orientation_bank_filters(pipe.orientations), (h // 2, w // 2))
    gray = _call_gray(torch, res)
    assert np.array_equal(gray, ref["gray"], equal_nan=True), name
    assert np.array_equal(_np(res.points), peak_reference(ref["gray"], 0.5)), name


@pytest.mark.gpu
@pytest.mark.parametrize("nb", (None, 4, 8, 12, 16))
def test_run_and_run_unfused_on_a_pyramid(nb, cuda):
    torch = cuda
    from pysilent_b200 import LineEndPipeline
    frames = torch.from_numpy(_bgr([("struct", 71), ("noise", 71, 0)], 96, 128)).cuda()
    for p in (0.0, 0.5, 0.9):
        pipe = LineEndPipeline(output_size=(48, 32), zoom_ratio=SQRT2, orientations=nb, peaks=p)
        pyr = pipe.plan_for(frames).build(frames)
        calls = [("run", pipe.run)] + ([("run_unfused", pipe.run_unfused)] if nb is None else [])
        for what, fn in calls:
            res = fn(pyr)
            assert res.gray is not None
            want = peak_reference(_np(res.gray), p)
            assert len(want) > 0 and np.array_equal(_np(res.points), want), (nb, p, what)
            assert np.array_equal(_np(res.gray), _call_gray(torch, res), equal_nan=True), (nb, p, what)
            assert fn(pyr, want_points=False).points is None


def _kernel_names(torch, fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type.name == "CUDA"]


def _count(names, kernel):
    return sum(kernel in n for n in names)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ("f32_480p_b3", "nv12_b3", "bank16_b3", "pyramid_float_b8"))
def test_profiler_shows_the_peak_kernels_only(name, cuda):
    torch = cuda
    pipe, frames, _ = _peak_pipe(torch, name, 0.5)
    names = _kernel_names(torch, lambda: pipe.run_frames(frames, points_capacity=1 << 20))
    emits = _count(names, "peak_write_kernel")   # (PYRAMID ignores the capacity: a short first buffer takes two emits)
    assert emits in (1, 2) and (emits == 1 or CASES[name][4] == "pyramid"), (name, emits)
    for k in PEAK_KERNELS:
        assert _count(names, k) == emits, (name, k, names)
    for k in REGION_KERNELS:
        assert _count(names, k) == 0, (name, k)
    region = _pipe(torch, *CASES[name][1:4])
    names = _kernel_names(torch, lambda: region.run_frames(frames))
    assert not any(_count(names, k) for k in ("peak_count_kernel", "peak_write_kernel", "peak_base_kernel"))
    assert any(_count(names, k) for k in REGION_KERNELS)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [{}, dict(orientations=8, out_dtype="f16"), dict(frame_format="nv12")],
                         ids=["f32", "bank8_f16", "nv12"])
def test_capacity_contract_and_emit_only_redo(kw, cuda):
    torch = cuda
    size, zoom, p = (96, 64), 1.3, 0.5
    if kw.get("frame_format") == "nv12":
        frames = torch.from_numpy(random_nv12(81, 480, 640, 3)).cuda()
    else:
        frames = torch.from_numpy(_bgr([("periodic", 12, 1), ("noise", 12, 0), ("struct", 3)], 480, 640)).cuda()
    pipe = _pipe(torch, size, zoom, dict(kw, peaks=p))
    full = pipe.run_frames(frames)
    pts = _np(full.points)
    total = len(pts)
    assert total > 100
    plan = pipe.plan_for(frames)
    c = full.orient.shape[-1]
    orient = torch.empty((3 * plan.levels, size[1], size[0], c), dtype=pipe.out_dtype, device="cuda")
    line_end = torch.empty_like(orient)
    for cap in (0, 1, total - 1, total):
        big = torch.full((total + 16, 4), SENTINEL, dtype=torch.int64, device="cuda")
        count = torch.full((1,), -1, dtype=torch.int64, device="cuda")
        out = (orient, line_end, big[:cap], count)
        pipe.run_frames(frames, out=out)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            res = pipe.run_frames(frames, out=out)
        finally:
            torch.cuda.set_sync_debug_mode(0)
        torch.cuda.synchronize()
        assert res.points.shape[0] == cap and int(count.item()) == total, (kw, cap)
        assert np.array_equal(_np(big)[:cap], pts[:cap]), (kw, cap)
        assert (_np(big)[cap:] == SENTINEL).all(), (kw, cap, "rows past the capacity")
        assert np.array_equal(_np(orient.float()), _np(full.orient.float()), equal_nan=True)
    # a capacity short of the total redoes only the emit: one pipeline, two peak emits
    for cap in (1, total - 1):
        names = _kernel_names(torch, lambda: pipe.run_frames(frames, points_capacity=cap))
        assert _count(names, "peak_write_kernel") == 2 and _count(names, "peak_count_kernel") == 2, cap
        assert _count(names, "stack_a_kernel") == 1, cap
        assert np.array_equal(_np(pipe.run_frames(frames, points_capacity=cap).points), pts), cap
    names = _kernel_names(torch, lambda: pipe.run_frames(frames, points_capacity=total))
    assert _count(names, "peak_write_kernel") == 1


@pytest.mark.gpu
@pytest.mark.parametrize("r", (None, 0, 2))
@pytest.mark.parametrize("name", ("f32_480p_b3", "nv12_b3", "bank12_b3", "bank8_f16_b1", "pyramid_w100_b12",
                                  "convert_nv12_w100_b4"))
def test_records_and_patches_of_peak_points(name, r, cuda):
    torch = cuda
    from pysilent_b200 import _ops
    pipe, frames, route = _peak_pipe(torch, name, 0.5)
    res = pipe.run_frames(frames)
    pts = res.points
    assert len(pts) > 0
    rec = pipe.run_frames_records(frames, patch_radius=r)
    assert np.array_equal(_np(rec.points), _np(pts)), name
    nv12 = pipe.frame_format == "nv12"
    batched = frames if frames.dim() == (3 if nv12 else 4) else frames.unsqueeze(0)
    H, W = (batched.shape[-2] * 2 // 3, batched.shape[-1]) if nv12 else batched.shape[-3:-1]
    make, size, zoom, _, _ = CASES[name]
    # gray: the call's own (PLAN: the plan's, of its latest call, which ran these frames)
    plan = _geometry_plan(H, W, size, zoom) if res.gray is not None else pipe.plan_for(batched)
    gray = res.gray
    count = torch.full((1,), len(pts), dtype=torch.int64, device="cuda")
    offs, yx, vals = _ops.point_records(plan, batched.shape[0], pts.contiguous(), count, res.orient, res.padded_line_end,
                                        gray, radius=r)
    want = PointRecords_of(offs, yx, vals)
    for field in ("frame_offsets", "frame_yx", "gray", "orient", "line_end"):
        g, w = _np(getattr(rec, field)), _np(want[field])
        assert g.shape == w.shape and np.array_equal(g, w, equal_nan=True), (name, r, field)


def PointRecords_of(offs, yx, vals):
    c = (vals.shape[-1] - 1) // 2
    return dict(frame_offsets=offs, frame_yx=yx, gray=vals[..., 0], orient=vals[..., 1:1 + c], line_end=vals[..., 1 + c:])


@pytest.mark.gpu
def test_records_out_buffers_take_no_host_synchronisation(cuda):
    torch = cuda
    size, zoom = (96, 64), 1.5
    pipe = _pipe(torch, size, zoom, dict(peaks=0.5))
    frames = torch.from_numpy(_bgr([("noise", 60, i) for i in range(3)], 240, 320)).cuda()
    L = pipe.plan_for(frames).levels
    cap = 64
    out = (torch.empty((3 * L, 64, 96, 3), device="cuda"), torch.empty((3 * L, 64, 96, 3), device="cuda"),
           torch.empty((cap, 4), dtype=torch.int64, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda"),
           torch.empty(4, dtype=torch.int64, device="cuda"), torch.empty((cap, 2), device="cuda"),
           torch.empty((cap, 5, 5, 7), device="cuda"))
    pipe.run_frames_records(frames, out=out, patch_radius=2)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        rec = pipe.run_frames_records(frames, out=out, patch_radius=2)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    want = pipe.run_frames_records(frames, patch_radius=2)
    total = len(want.points)
    assert int(out[3].item()) == total > cap
    assert np.array_equal(_np(rec.points), _np(want.points)[:cap])
    assert np.array_equal(_np(rec.gray), _np(want.gray)[:cap], equal_nan=True)
    assert np.array_equal(_np(rec.frame_offsets), np.minimum(_np(want.frame_offsets), cap))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12", "bgr_f16", "bank8"])
def test_host_entry_points_equal_the_device_calls(fmt, cuda):
    torch = cuda
    size, zoom = (288, 192), 1.3
    if fmt == "nv12":
        frames = random_nv12(91, 480, 640, 3)
        kw = dict(frame_format="nv12")
    else:
        frames = _bgr([("noise", 92, 0), ("struct", 92), ("noise", 92, 1)], 480, 640)
        kw = dict(out_dtype="f16") if fmt == "bgr_f16" else (dict(orientations=8) if fmt == "bank8" else {})
    pipe = _pipe(torch, size, zoom, dict(kw, peaks=0.5))
    dev = pipe.run_frames(torch.from_numpy(frames).cuda())
    pts = _np(dev.points)
    assert len(pts) > 100
    host = pipe.run_host(frames, points_capacity=8)   # also redoes the emit with room for every point
    assert isinstance(host.points, np.ndarray) and np.array_equal(host.points, pts), fmt
    assert np.array_equal(host.orient, _np(dev.orient), equal_nan=True)
    assert np.array_equal(host.padded_line_end, _np(dev.padded_line_end), equal_nan=True)
    want = pipe.run_frames_records(torch.from_numpy(frames).cuda(), patch_radius=4)
    got = pipe.run_host_records(frames, points_capacity=8, patch_radius=4)
    for field in got._fields:
        g = getattr(got, field)
        assert isinstance(g, np.ndarray) and np.array_equal(g, _np(getattr(want, field)), equal_nan=True), (fmt, field)
    plain = pipe.run_host_records(frames)
    assert np.array_equal(plain.points, pts)
    if fmt != "bank8":
        cb = pipe.callback(frames[0])
        first = int(np.searchsorted(pts[:, 0], len(cb[1])))
        assert np.array_equal(cb[3], pts[:first]), fmt
        assert len(cb[1]) == len(dev.orient) // len(frames)


@pytest.mark.gpu
def test_peaks_none_keeps_the_region_maxima(cuda):
    torch = cuda
    from pysilent_b200 import LineEndPipeline
    frames = _bgr([("struct", 95), ("noise", 95, 0)], 240, 320)
    a = LineEndPipeline(output_size=(96, 64), zoom_ratio=1.5)
    b = LineEndPipeline(output_size=(96, 64), zoom_ratio=1.5, peaks=None)
    ra, rb = a.run_host(frames), b.run_host(frames)
    assert len(ra.points) > 0 and np.array_equal(ra.points, rb.points)
    peaks = LineEndPipeline(output_size=(96, 64), zoom_ratio=1.5, peaks=0.5).run_host(frames)
    assert len(peaks.points) > 4 * len(peaks.orient)
    assert np.array_equal(peaks.orient, ra.orient, equal_nan=True)
