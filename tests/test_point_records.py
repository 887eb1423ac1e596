"""Feature-point records (``silent_point_records``, ``LineEndPipeline.run_frames_records`` / ``run_host_records``).

A record holds a point's frame position and the responses at it. The position follows scipy.ndimage.zoom's sample
position per axis, ``offset + o * (n_in - 1) / (n_out - 1)`` in float64, rounded once to float32. It is NaN where the
tap tables define the row or column as 0. The CPU tests check the plan's coordinate tables against a numpy restatement
of that rule, and the rule itself against scipy. They also check every argument check of the C call and of the Python
entry points. The GPU tests check the records bit for bit against the call's own outputs indexed at the points, on every
route, and check the capacity contract.
"""
import ctypes

import numpy as np
import pytest

from conftest import structured_frame, synthetic_frame
from pysilent_b200 import _lib

SQRT2 = 2 ** .5
SENTINEL = -0x5EE7
FSENTINEL = -12345.5


def _geometry_plan(H, W, center, scale):
    """A plan of H x W frames: its geometry is that of every frame dtype and format of that size."""
    import torch
    from pysilent_b200.util.zoom.from_image import PyramidPlan
    return PyramidPlan((H, W, 3), torch.uint8, 3, center, scale)


# ---- CPU: the coordinate rule --------------------------------------------------------------------------------------------

# frame (H, W), output_size (w, h), zoom
GEOMETRY_CASES = {
    "480p_1.3": ((480, 640), (288, 192), 1.3),
    "720p_sqrt2": ((720, 1280), (288, 192), SQRT2),
    "1080p_sqrt2": ((1080, 1920), (288, 192), SQRT2),
    "4k_sqrt2": ((2160, 3840), (288, 192), SQRT2),
    "odd_301x517": ((301, 517), (97, 61), 1.37),
    "odd_255x333": ((255, 333), (51, 41), 1.21),
}


def restated_axis(info_lo, info_hi, valid, n_keep, scale, level):
    """The coordinate rule of one axis of one level, restated in numpy: float32(lo + o * factor), NaN where o >= valid
    or the position leaves [0, n_in - 1]."""
    n_in = info_hi - info_lo
    out = np.full(n_keep, np.nan, np.float32)
    if n_in <= 0:
        return out
    n_out = int(round(n_in * (1.0 / scale ** level)))   # scipy's int(round(in * zoom)), half to even
    factor = (n_in - 1) / (n_out - 1) if n_out > 1 else 1.0
    for o in range(min(valid, n_keep)):
        cc = o * factor
        if 0 <= cc <= n_in - 1:
            out[o] = np.float32(info_lo + cc)
    return out


def _restated(plan, scale, level):
    y0, y1, x0, x1, vh, vw = plan.level_info(level)
    return (restated_axis(y0, y1, vh, plan.h, scale, level), restated_axis(x0, x1, vw, plan.w, scale, level))


def _same_bits(got, want):
    got, want = np.asarray(got), np.asarray(want)
    return got.shape == want.shape and np.array_equal(np.isnan(got), np.isnan(want)) and \
        np.array_equal(np.where(np.isnan(got), 0, got).view(np.uint32), np.where(np.isnan(want), 0, want).view(np.uint32))


def test_symbols_exported_and_bound(built_lib):
    for name in ("silent_point_records", "silent_plan_level_coords"):
        assert name in _lib.SYMBOLS and hasattr(built_lib, name), name
        assert getattr(built_lib, name).argtypes, name


@pytest.mark.parametrize("case", sorted(GEOMETRY_CASES))
def test_plan_coordinates_equal_the_restated_rule(case, built_lib):
    (H, W), center, scale = GEOMETRY_CASES[case]
    plan = _geometry_plan(H, W, center, scale)
    assert plan.levels > 0
    tail_zero = False
    for level in range(plan.levels):
        fy, fx = plan.level_coords(level)
        iy, _, ix, _ = plan.level_tables(level)
        ry, rx = _restated(plan, scale, level)
        # NaN exactly where the tap tables define the row / column as 0, the restated value bit for bit elsewhere
        assert np.array_equal(np.isnan(fy), iy[:, 0] < 0) and np.array_equal(np.isnan(fx), ix[:, 0] < 0), (case, level)
        assert _same_bits(fy, ry) and _same_bits(fx, rx), (case, level)
        tail_zero |= bool(np.isnan(fy).any())
    if case == "1080p_sqrt2":
        assert tail_zero, "1080p at sqrt(2): the last level's tail row (o >= valid_h) is defined as 0"
    if case == "4k_sqrt2":
        assert plan.levels == 8


@pytest.mark.parametrize("case", sorted(GEOMETRY_CASES))
def test_restated_rule_against_scipy_zoom(case):
    """On a frame that holds its own column (row) index, scipy.ndimage.zoom(order=5, prefilter=False) reproduces the
    linear ramp away from the mirrored edges: the zoomed level holds the restated coordinate there."""
    ndimage = pytest.importorskip("scipy.ndimage")
    (H, W), center, scale = GEOMETRY_CASES[case]
    plan = _geometry_plan(H, W, center, scale)
    checked = 0
    for level in range(plan.levels):
        info = plan.level_info(level)
        for lo, hi, coords in ((info[0], info[1], _restated(plan, scale, level)[0]),
                               (info[2], info[3], _restated(plan, scale, level)[1])):
            n_in = hi - lo
            zoomed = ndimage.zoom(np.arange(lo, hi, dtype=np.float64), 1.0 / scale ** level, order=5, prefilter=False)
            n = min(len(zoomed), len(coords))
            o = np.arange(n)
            cc = coords[:n].astype(np.float64) - lo
            inner = ~np.isnan(coords[:n]) & (cc >= 3) & (cc <= n_in - 4)
            tol = np.spacing(np.abs(coords[:n][inner]).astype(np.float32)).astype(np.float64)
            assert (np.abs(zoomed[o[inner]] - coords[:n][inner]) <= tol).all(), (case, level)
            checked += int(inner.sum())
    assert checked > 0


# ---- CPU: argument checks ------------------------------------------------------------------------------------------------

def _raw_plan(L, H=240, W=320, center=(96, 64), scale=1.5):
    p = _lib.SilentParams(H, W, 3, 3, center[0], center[1], float(scale), _lib.SILENT_U8, 0)
    h = ctypes.c_void_p()
    assert L.silent_plan_create(ctypes.byref(p), ctypes.byref(h)) == 0, L.silent_last_error()
    return h


def test_status_codes_before_any_cuda_call(built_lib):
    """Every check fails on the host: these calls reach no CUDA call, with or without a device (the plan is never
    reserved, so the plan's gray cannot be read)."""
    L = built_lib
    plan = _raw_plan(L)
    zero = _raw_plan(L, H=64, W=96, center=(96, 64))   # frame no larger than the centre: 0 levels
    assert L.silent_plan_levels(zero) == 0
    fake = ctypes.c_void_p(256)
    good = dict(plan=plan, batch=1, points=fake, count=fake, capacity=8, orient=fake, line_end=fake, channels=3, half=0,
                gray=fake, offsets=fake, coords=fake, values=fake)

    def call(**kw):
        a = dict(good, **kw)
        return L.silent_point_records(a["plan"], a["batch"], a["points"], a["count"], a["capacity"], a["orient"],
                                      a["line_end"], a["channels"], a["half"], a["gray"], a["offsets"], a["coords"],
                                      a["values"], None)
    try:
        for kw in (dict(plan=None), dict(count=None), dict(orient=None), dict(line_end=None), dict(offsets=None),
                   dict(points=None), dict(coords=None), dict(values=None), dict(capacity=-1), dict(half=2),
                   dict(batch=0), dict(batch=-3)):
            assert call(**kw) == _lib_status("INVAL"), kw
        for ch in (0, 1, 2, 5, 6, 7, 9, 15, 17, 32):
            assert call(channels=ch) == _lib_status("SHAPE"), ch
        assert call(plan=zero) == _lib_status("SHAPE")
        assert call(gray=None) == _lib_status("CAPACITY")            # the plan's gray: no frames reserved
        assert call(gray=None, batch=5, channels=16, half=1) == _lib_status("CAPACITY")
        assert b"reserve" in L.silent_last_error()
        # capacity 0 needs no points, coords or values (checks still fail on the unreserved plan's gray)
        assert call(capacity=0, points=None, coords=None, values=None, gray=None) == _lib_status("CAPACITY")
        assert L.silent_plan_level_coords(None, 0, None, None) == _lib_status("INVAL")
        assert L.silent_plan_level_coords(plan, L.silent_plan_levels(plan), None, None) == _lib_status("INVAL")
        assert L.silent_plan_level_coords(plan, -1, None, None) == _lib_status("INVAL")
    finally:
        L.silent_plan_destroy(plan)
        L.silent_plan_destroy(zero)


def _lib_status(name):
    return dict(INVAL=-1, SHAPE=-2, CAPACITY=-3, CUDA=-4)[name]


def test_python_validation_raises_before_the_gpu():
    import torch
    from pysilent_b200 import LineEndPipeline, _ops
    frames = torch.zeros((1, 48, 64, 3), dtype=torch.uint8)
    for nb in (1, 2, 5, 6, 7):
        with pytest.raises(ValueError, match="records need"):
            LineEndPipeline(output_size=(34, 18), zoom_ratio=SQRT2, orientations=nb).run_frames_records(frames)
    with pytest.raises(ValueError):
        LineEndPipeline(orientations=20).run_frames_records(frames)
    pipe = LineEndPipeline(output_size=(34, 18), zoom_ratio=SQRT2)
    with pytest.raises(ValueError, match="points_capacity"):
        pipe.run_frames_records(frames, points_capacity=-1)
    o = torch.zeros((2, 18, 34, 3))
    with pytest.raises(ValueError, match="takes"):
        pipe.run_frames_records(frames, out=(o, o, torch.zeros((4, 4), dtype=torch.int64), torch.zeros(1)))
    with pytest.raises(ValueError, match="float16"):
        LineEndPipeline(output_size=(34, 18), zoom_ratio=SQRT2, out_dtype=torch.float16).run_frames_records(
            frames, out=(o, o) + (None,) * 5)

    plan = _geometry_plan(48, 64, (34, 18), SQRT2)
    n = plan.levels
    pts, cnt = torch.zeros((4, 4), dtype=torch.int64), torch.zeros(1, dtype=torch.int64)
    o = torch.zeros((n, 18, 34, 3))
    bad = [dict(batch=0), dict(orient=torch.zeros((n + 1, 18, 34, 3))), dict(orient=torch.zeros((n, 18, 34, 5)),
           line_end=torch.zeros((n, 18, 34, 5))), dict(line_end=o.half()), dict(orient=o.double(), line_end=o.double()),
           dict(points=torch.zeros((4, 3), dtype=torch.int64)), dict(points=pts.int()), dict(count=cnt.float()),
           dict(gray=torch.zeros((n, 18, 34, 3))), dict(frame_offsets=torch.zeros(3, dtype=torch.int64)),
           dict(frame_yx=torch.zeros((4, 3))), dict(values=torch.zeros((4, 6))), {}]   # {}: CPU tensors
    for kw in bad:
        a = dict(batch=1, points=pts, count=cnt, orient=o, line_end=o)
        a.update(kw)
        with pytest.raises(ValueError):
            _ops.point_records(plan, **a)


# ---- GPU -----------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cuda(built_lib):
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def random_nv12(seed, h, w, batch):
    return np.random.RandomState(seed).randint(0, 256, size=(batch, h * 3 // 2, w)).astype(np.uint8)


def periodic_frame(p, seed, h, w):
    tile = np.random.RandomState(seed).randint(0, 256, size=(p, p, 3)).astype(np.uint8)
    return np.ascontiguousarray(np.tile(tile, (h // p + 1, w // p + 1, 1))[:h, :w])


def _bgr(specs, h, w):
    out = []
    for s in specs:
        if s[0] == "noise":
            out.append(synthetic_frame(s[1], s[2], h, w))
        elif s[0] == "struct":
            out.append(structured_frame(s[1], h, w))
        else:
            out.append(periodic_frame(s[1], s[2], h, w))
    return np.stack(out)


# name: (frames maker, output_size, zoom, pipeline keywords, route)
def _cases():
    c = {
        "f32_480p_b3": (lambda: _bgr([("noise", 41, i) for i in range(3)], 480, 640), (288, 192), 1.3, {}, "plan"),
        "f16_480p_b3": (lambda: _bgr([("noise", 42, i) for i in range(3)], 480, 640), (288, 192), 1.3,
                        dict(out_dtype="f16"), "plan"),
        "single_720p": (lambda: synthetic_frame(43, 0, 720, 1280), (288, 192), SQRT2, {}, "plan"),
        "struct_b3": (lambda: _bgr([("struct", 44), ("noise", 44, 0), ("struct", 45)], 240, 320), (96, 64), 1.5, {},
                      "plan"),
        "struct_1080p_b2": (lambda: _bgr([("struct", 46), ("noise", 46, 1)], 1080, 1920), (288, 192), SQRT2,
                            dict(out_dtype="f16"), "plan"),
        "nv12_b3": (lambda: random_nv12(47, 240, 320, 3), (96, 64), 1.5, dict(frame_format="nv12"), "plan"),
        "nv12_f16_b1": (lambda: random_nv12(48, 480, 640, 1), (288, 192), 1.3,
                        dict(frame_format="nv12", out_dtype="f16"), "plan"),
        "4k_b2_8levels": (lambda: _bgr([("noise", 49, 0), ("struct", 49)], 2160, 3840), (288, 192), SQRT2, {}, "plan"),
        "4k_b1_bank16": (lambda: _bgr([("noise", 50, 0)], 2160, 3840), (288, 192), SQRT2, dict(orientations=16),
                         "plan"),
        # PYRAMID: float frames with a bank; uint8 rows of 300 bytes (not 16-byte multiples) with banks of 12 and 8
        "pyramid_float_b8": (lambda: (_bgr([("noise", 51, i) for i in range(3)], 96, 128) / 3.0).astype(np.float32),
                             (48, 32), SQRT2, dict(orientations=8), "pyramid"),
        "pyramid_w100_b12": (lambda: _bgr([("noise", 52, i) for i in range(3)], 72, 100), (34, 18), SQRT2,
                             dict(orientations=12), "pyramid"),
        "pyramid_w100_b8_f16": (lambda: _bgr([("struct", 53), ("noise", 53, 0)], 72, 100), (34, 18), SQRT2,
                                dict(orientations=8, out_dtype="f16"), "pyramid"),
        # CONVERT: NV12 frames whose BGR rows are not 16-byte multiples, with a bank -> BGR on the GPU -> PYRAMID
        "convert_nv12_w100_b4": (lambda: random_nv12(54, 72, 100, 3), (34, 18), SQRT2,
                                 dict(orientations=4, frame_format="nv12"), "convert"),
    }
    for nb in (4, 8, 12, 16):
        c["bank%d_b3" % nb] = (lambda nb=nb: _bgr([("periodic", 4, nb), ("noise", 55, nb), ("struct", nb)], 96, 128),
                               (48, 32), SQRT2, dict(orientations=nb), "plan")
        c["bank%d_f16_b1" % nb] = (lambda nb=nb: _bgr([("noise", 56, nb)], 96, 128), (48, 32), SQRT2,
                                   dict(orientations=nb, out_dtype="f16"), "plan")
    return c


CASES = _cases()


def _pipe(torch, size, zoom, kw):
    from pysilent_b200 import LineEndPipeline
    kw = dict(kw)
    if kw.get("out_dtype") == "f16":
        kw["out_dtype"] = torch.float16
    return LineEndPipeline(output_size=size, zoom_ratio=zoom, **kw)


def _np(t):
    return t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)


def _assert_bits(got, want, what):
    got, want = _np(got), np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    same = (got == want) | (np.isnan(got) & np.isnan(want))
    assert same.all(), "%s: %d of %d values differ" % (what, (~same).sum(), same.size)


def _frame_hw(frames, nv12):
    return (frames.shape[-2] * 2 // 3, frames.shape[-1]) if nv12 else frames.shape[-3:-1]


def _expected(torch, pipe, frames_dev, size, zoom):
    """What the records must hold: run_frames's own outputs indexed at its points, the gray of the same stack, the
    plan's coordinate tables and the per-frame search of the points."""
    from pysilent_b200 import _ops
    nv12 = pipe.frame_format == "nv12"
    res = pipe.run_frames(frames_dev)
    pts = _np(res.points)
    gray = res.gray
    if gray is None:   # PLAN: the pipeline keeps gray in its plan; the stack on the plan's NHWC pyramid gives it
        batched = frames_dev if frames_dev.dim() == (3 if nv12 else 4) else frames_dev.unsqueeze(0)
        pyr = pipe.plan_for(batched).build(batched.contiguous())
        gray = (_ops.stack_fused(pyr, pipe.stack_weights())[2] if pipe.orientations is None
                else _ops.stack_bank(pyr, pipe.orientation_bank())[2])
    H, W = _frame_hw(frames_dev, nv12)
    plan = _geometry_plan(H, W, size, zoom)
    L = plan.levels
    b = res.orient.shape[0] // L
    fy = np.stack([plan.level_coords(l)[0] for l in range(L)])
    fx = np.stack([plan.level_coords(l)[1] for l in range(L)])
    n, y, x = pts[:, 0], pts[:, 1], pts[:, 2]
    orient, line_end, gray = _np(res.orient.float()), _np(res.padded_line_end.float()), _np(gray)
    return dict(points=pts, frame_offsets=np.searchsorted(pts[:, 0], np.arange(b + 1) * L, side="left"),
                frame_yx=np.stack([fy[n % L, y], fx[n % L, x]], axis=1).astype(np.float32),
                gray=gray[n, y, x, 0], orient=orient[n, y, x], line_end=line_end[n, y, x], levels=L, batch=b)


def _check(rec, want, what):
    assert _np(rec.points).dtype == np.int64 and np.array_equal(_np(rec.points), want["points"]), what + " points"
    assert np.array_equal(_np(rec.frame_offsets), want["frame_offsets"]), what + " frame_offsets"
    for field in ("frame_yx", "gray", "orient", "line_end"):
        assert _np(getattr(rec, field)).dtype == np.float32, (what, field)
        _assert_bits(getattr(rec, field), want[field], "%s %s" % (what, field))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_records_equal_the_calls_own_outputs(name, cuda):
    torch = cuda
    make, size, zoom, kw, route = CASES[name]
    pipe = _pipe(torch, size, zoom, kw)
    frames = torch.from_numpy(make()).cuda()
    nv12 = pipe.frame_format == "nv12"
    batched = frames if frames.dim() == (3 if nv12 else 4) else frames.unsqueeze(0)
    from pysilent_b200.pipeline import CONVERT, PLAN, PYRAMID
    nb = pipe.orientations
    got_route = pipe._frame_route(nb, pipe.frame_format, batched.dtype, batched.shape)
    assert got_route == dict(plan=PLAN, pyramid=PYRAMID, convert=CONVERT)[route], (name, got_route)
    want = _expected(torch, pipe, frames, size, zoom)
    assert len(want["points"]) > 0, name
    rec = pipe.run_frames_records(frames)
    _check(rec, want, name)
    assert rec.orient.shape[1] == (nb or 3)


def _capacities(pts, offsets):
    total = len(pts)
    same_row = np.nonzero((pts[1:, :2] == pts[:-1, :2]).all(axis=1))[0] + 1
    inner_edges = [int(o) for o in offsets[1:-1] if 0 < o < total]
    return dict(zero=0, one=1, total_minus_1=total - 1, total=total, in_run=int(same_row[len(same_row) // 2]),
                frame_edge=inner_edges[0])


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [{}, dict(orientations=8, out_dtype="f16")], ids=["f32", "bank8_f16"])
def test_capacity_contract(kw, cuda):
    torch = cuda
    size, zoom = (96, 64), 1.3
    frames = torch.from_numpy(_bgr([("periodic", 12, 1), ("noise", 12, 0), ("struct", 3)], 480, 640)).cuda()
    pipe = _pipe(torch, size, zoom, kw)
    full = pipe.run_frames_records(frames)
    pts, offsets = _np(full.points), _np(full.frame_offsets)
    total = len(pts)
    caps = _capacities(pts, offsets)
    assert 1 < caps["in_run"] < total - 1 and 1 < caps["frame_edge"] < total - 1, caps
    assert (pts[caps["in_run"], :2] == pts[caps["in_run"] - 1, :2]).all()
    c = full.orient.shape[1]
    L = pipe.plan_for(frames).levels
    dt = pipe.out_dtype
    orient = torch.empty((3 * L, size[1], size[0], c), dtype=dt, device="cuda")
    line_end = torch.empty_like(orient)
    for kind, cap in caps.items():
        big_pts = torch.full((total + 16, 4), SENTINEL, dtype=torch.int64, device="cuda")
        big_yx = torch.full((total + 16, 2), FSENTINEL, dtype=torch.float32, device="cuda")
        big_val = torch.full((total + 16, 1 + 2 * c), FSENTINEL, dtype=torch.float32, device="cuda")
        offs = torch.full((4,), SENTINEL, dtype=torch.int64, device="cuda")
        count = torch.full((1,), -1, dtype=torch.int64, device="cuda")
        rec = pipe.run_frames_records(frames, out=(orient, line_end, big_pts[:cap], count, offs, big_yx[:cap],
                                                   big_val[:cap]))
        torch.cuda.synchronize()
        what = "%s cap %s=%d" % (kw, kind, cap)
        assert int(count.item()) == total, what
        assert rec.points.shape[0] == cap and rec.frame_yx.shape[0] == cap, what
        assert np.array_equal(_np(big_pts)[:cap], pts[:cap]), what
        _assert_bits(_np(big_yx)[:cap], _np(full.frame_yx)[:cap], what + " frame_yx")
        vals = np.concatenate([_np(full.gray)[:, None], _np(full.orient), _np(full.line_end)], axis=1)
        _assert_bits(_np(big_val)[:cap], vals[:cap], what + " values")
        assert (_np(big_pts)[cap:] == SENTINEL).all(), what + ": points past the capacity"
        assert (_np(big_yx)[cap:] == FSENTINEL).all() and (_np(big_val)[cap:] == FSENTINEL).all(), \
            what + ": records past the capacity"
        assert np.array_equal(_np(offs), np.minimum(offsets, cap)), what + " frame_offsets"


@pytest.mark.gpu
def test_out_buffers_take_no_host_synchronisation(cuda):
    torch = cuda
    size, zoom = (96, 64), 1.5
    pipe = _pipe(torch, size, zoom, {})
    frames = torch.from_numpy(_bgr([("noise", 60, i) for i in range(3)], 240, 320)).cuda()
    L = pipe.plan_for(frames).levels
    cap = 512
    out = (torch.empty((3 * L, 64, 96, 3), device="cuda"), torch.empty((3 * L, 64, 96, 3), device="cuda"),
           torch.empty((cap, 4), dtype=torch.int64, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda"),
           torch.empty(4, dtype=torch.int64, device="cuda"), torch.empty((cap, 2), device="cuda"),
           torch.empty((cap, 7), device="cuda"))
    pipe.run_frames_records(frames, out=out)   # plan set-up and workspace outside the checked call
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        rec = pipe.run_frames_records(frames, out=out)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    total = int(out[3].item())
    assert 0 < total <= cap
    want = pipe.run_frames_records(frames)
    assert np.array_equal(_np(rec.points)[:total], _np(want.points))
    _assert_bits(_np(rec.orient)[:total], _np(want.orient), "orient")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12", "bgr_f16"])
def test_host_records_equal_device_records(fmt, cuda):
    torch = cuda
    size, zoom = (288, 192), 1.3
    if fmt == "nv12":
        frames = random_nv12(61, 480, 640, 3)
        kw = dict(frame_format="nv12")
    else:
        frames = _bgr([("noise", 62, i) for i in range(3)], 480, 640)
        kw = dict(out_dtype="f16") if fmt == "bgr_f16" else {}
    pipe = _pipe(torch, size, zoom, kw)
    want = pipe.run_frames_records(torch.from_numpy(frames).cuda())
    pinned = torch.empty(frames.shape, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[...] = frames
    for what, src in (("pageable", frames), ("pinned", pinned.numpy())):
        got = pipe.run_host_records(src, points_capacity=8)   # also redoes the call with room for every point
        for field in got._fields:
            assert isinstance(getattr(got, field), np.ndarray), (what, field)
            _assert_bits(getattr(got, field), _np(getattr(want, field)), "%s %s %s" % (fmt, what, field))
    single = pipe.run_host_records(frames[0])
    first = _np(want.frame_offsets)[1]
    assert np.array_equal(single.points, _np(want.points)[:first]) and list(single.frame_offsets) == [0, first]
