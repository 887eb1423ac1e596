"""Feature-point patches (``silent_point_patches``, ``run_frames_records`` / ``run_host_records`` with
``patch_radius``).

A patch of radius r holds, for each point (level, y, x), the values of gray, orient[C] and line_end[C] at (y + dy,
x + dx) for dy, dx in [-r, r], at [r + dy][r + dx], and +0.0 where that pixel leaves the level. The CPU tests check the
binding, every status code of the C call and the Python validation. The GPU tests check the patches bit for bit against
a numpy zero-padded slice of the call's own outputs on every route the records serve, the borders of a level, the
capacity contract, the absence of host synchronisation with ``out=`` and the host entry point against the device one.
"""
import ctypes
import os

import numpy as np
import pytest

from test_point_records import (CASES, FSENTINEL, SENTINEL, SQRT2, _bgr, _capacities, _geometry_plan, _lib_status, _np,
                                _pipe, _raw_plan, random_nv12)
from pysilent_b200 import _lib

RADII = (0, 1, 4)
BAD_RADII = (-1, 32, -100, 1000, 1.0, 2.5, True, False, "1", np.float32(2))


def _same_bits(got, want, what):
    """Equal bit patterns (so +0.0 and -0.0 differ) and the same NaN mask."""
    got, want = _np(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype == np.float32, (what, got.shape, want.shape, got.dtype)
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    assert np.array_equal(nan_g, nan_w), "%s: NaN masks differ at %d values" % (what, (nan_g != nan_w).sum())
    differ = (got.view(np.uint32) != want.view(np.uint32)) & ~nan_g
    assert not differ.any(), "%s: %d of %d values differ" % (what, differ.sum(), got.size)


def zero_padded_patches(arr, pts, r):
    """``arr`` [N, h, w] or [N, h, w, C] sliced around each row (n, y, x) of ``pts`` after zero padding by r:
    [K, P, P] or [K, P, P, C]."""
    a = np.pad(arr, [(0, 0), (r, r), (r, r)] + [(0, 0)] * (arr.ndim - 3))
    d = np.arange(2 * r + 1)
    n, y, x = pts[:, 0], pts[:, 1], pts[:, 2]
    return a[n[:, None, None], (y[:, None] + d)[:, :, None], (x[:, None] + d)[:, None, :]]


# ---- CPU -----------------------------------------------------------------------------------------------------------------

def test_symbol_exported_and_bound(built_lib):
    assert "silent_point_patches" in _lib.SYMBOLS and hasattr(built_lib, "silent_point_patches")
    assert len(built_lib.silent_point_patches.argtypes) == 15
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                               "silent_b200.h")).read()
    assert "#define SILENT_PATCH_RADIUS_MAX %d" % _lib.PATCH_RADIUS_MAX in header


def test_status_codes_before_any_cuda_call(built_lib):
    """Every check fails on the host: no call here reaches CUDA, with or without a device (the plan is never reserved,
    so a call that passes every other check fails on the plan's gray)."""
    L = built_lib
    plan = _raw_plan(L)
    zero = _raw_plan(L, H=64, W=96, center=(96, 64))   # frame no larger than the centre: 0 levels
    fake = ctypes.c_void_p(256)
    good = dict(plan=plan, batch=1, points=fake, count=fake, capacity=8, orient=fake, line_end=fake, channels=3, half=0,
                gray=fake, radius=2, offsets=fake, coords=fake, values=fake)

    def call(**kw):
        a = dict(good, **kw)
        return L.silent_point_patches(a["plan"], a["batch"], a["points"], a["count"], a["capacity"], a["orient"],
                                      a["line_end"], a["channels"], a["half"], a["gray"], a["radius"], a["offsets"],
                                      a["coords"], a["values"], None)
    try:
        for kw in (dict(plan=None), dict(count=None), dict(orient=None), dict(line_end=None), dict(offsets=None),
                   dict(points=None), dict(coords=None), dict(values=None), dict(capacity=-1), dict(half=2),
                   dict(batch=0), dict(batch=-3)):
            assert call(**kw) == _lib_status("INVAL"), kw
        for ch in (0, 1, 2, 5, 6, 7, 9, 15, 17, 32):
            assert call(channels=ch) == _lib_status("SHAPE"), ch
        for r in (-1, 32, -(2 ** 31), 2 ** 31 - 1):
            assert call(radius=r) == _lib_status("SHAPE"), r
            assert b"radius" in L.silent_last_error()
        assert call(plan=zero) == _lib_status("SHAPE")
        for r in (0, 1, 31):   # in range: the call goes on to the next check
            assert call(radius=r, gray=None) == _lib_status("CAPACITY"), r
            assert b"silent_point_patches" in L.silent_last_error()
        assert call(gray=None, batch=5, channels=16, half=1) == _lib_status("CAPACITY")
        assert call(capacity=0, points=None, coords=None, values=None, gray=None) == _lib_status("CAPACITY")
    finally:
        L.silent_plan_destroy(plan)
        L.silent_plan_destroy(zero)


def test_python_validation_raises_before_the_gpu():
    import torch
    from pysilent_b200 import LineEndPipeline, _ops
    assert _ops.patch_radius(None) is None and _ops.patch_radius(np.int64(3)) == 3 and _ops.patch_radius(31) == 31
    frames = torch.zeros((1, 48, 64, 3), dtype=torch.uint8)
    pipe = LineEndPipeline(output_size=(34, 18), zoom_ratio=SQRT2)
    for bad in BAD_RADII:
        with pytest.raises(ValueError, match="patch radius"):
            _ops.patch_radius(bad)
        with pytest.raises(ValueError, match="patch radius"):
            pipe.run_frames_records(frames, patch_radius=bad)
        with pytest.raises(ValueError, match="patch radius"):
            pipe.run_host_records(frames.numpy(), patch_radius=bad)

    # out=: the seventh buffer is [capacity, P, P, 1 + 2C] with a radius; all three record buffers are checked first
    plan = _geometry_plan(48, 64, (34, 18), SQRT2)
    n, cap = plan.levels, 6
    o = torch.zeros((n, 18, 34, 3))
    pts, cnt = torch.zeros((cap, 4), dtype=torch.int64), torch.zeros(1, dtype=torch.int64)
    offs, yx = torch.zeros(2, dtype=torch.int64), torch.zeros((cap, 2))
    good = torch.zeros((cap, 5, 5, 7))
    for kw in (dict(values=torch.zeros((cap, 7))), dict(values=torch.zeros((cap, 3, 3, 7))),
               dict(values=torch.zeros((cap + 1, 5, 5, 7))), dict(values=torch.zeros((cap, 5, 5, 9))),
               dict(values=good.double()), dict(values=None), dict(offs=torch.zeros(3, dtype=torch.int64)),
               dict(yx=torch.zeros((cap, 3))), dict(offs=offs.int())):
        a = dict(values=good, offs=offs, yx=yx)
        a.update(kw)
        with pytest.raises(ValueError):
            pipe.run_frames_records(frames, out=(o, o, pts, cnt, a["offs"], a["yx"], a["values"]), patch_radius=2)
    bank = LineEndPipeline(output_size=(34, 18), zoom_ratio=SQRT2, orientations=8)
    with pytest.raises(ValueError, match="values"):   # C = 8: 17 values per pixel
        bank.run_frames_records(frames, out=(o, o, pts, cnt, offs, yx, good), patch_radius=2)

    for kw in (dict(radius=-1), dict(radius=True), dict(radius=2, values=torch.zeros((4, 7))),
               dict(radius=0, values=torch.zeros((4, 7))), dict(values=torch.zeros((4, 1, 1, 7))),
               dict(radius=1, values=torch.zeros((4, 3, 3, 7)))):   # the last: CPU tensors
        a = dict(batch=1, points=torch.zeros((4, 4), dtype=torch.int64), count=cnt, orient=o, line_end=o)
        a.update(kw)
        with pytest.raises(ValueError):
            _ops.point_records(plan, **a)


# ---- GPU -----------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cuda(built_lib):
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


_OUTPUTS = {}


def _outputs(torch, name):
    """The case's pipeline, device frames and run_frames outputs as numpy: points, orient and line_end widened to
    float32, and gray [N, h, w] of the same stack."""
    if name not in _OUTPUTS:
        from pysilent_b200 import _ops
        make, size, zoom, kw, _ = CASES[name]
        pipe = _pipe(torch, size, zoom, kw)
        frames = torch.from_numpy(make()).cuda()
        nv12 = pipe.frame_format == "nv12"
        res = pipe.run_frames(frames)
        gray = res.gray
        if gray is None:   # PLAN: the pipeline keeps gray in its plan; the stack on the plan's NHWC pyramid gives it
            batched = (frames if frames.dim() == (3 if nv12 else 4) else frames.unsqueeze(0)).contiguous()
            pyr = pipe.plan_for(batched).build(batched)
            gray = (_ops.stack_fused(pyr, pipe.stack_weights())[2] if pipe.orientations is None
                    else _ops.stack_bank(pyr, pipe.orientation_bank())[2])
        _OUTPUTS[name] = (pipe, frames, dict(points=_np(res.points), orient=_np(res.orient.float()),
                                             line_end=_np(res.padded_line_end.float()), gray=_np(gray)[..., 0]))
    return _OUTPUTS[name]


def _check_patches(rec, out, r, what):
    pts = out["points"]
    assert np.array_equal(_np(rec.points), pts), what + " points"
    p = 2 * r + 1
    c = out["orient"].shape[-1]
    assert tuple(rec.gray.shape) == (len(pts), p, p) and tuple(rec.orient.shape) == (len(pts), p, p, c), what
    for field, arr in (("gray", out["gray"]), ("orient", out["orient"]), ("line_end", out["line_end"])):
        _same_bits(getattr(rec, field), zero_padded_patches(arr, pts, r), "%s %s" % (what, field))


@pytest.mark.gpu
@pytest.mark.parametrize("r", RADII)
@pytest.mark.parametrize("name", sorted(CASES))
def test_patches_equal_zero_padded_slices_of_the_calls_outputs(name, r, cuda):
    torch = cuda
    pipe, frames, out = _outputs(torch, name)
    assert len(out["points"]) > 0, name
    rec = pipe.run_frames_records(frames, patch_radius=r)
    what = "%s r=%d" % (name, r)
    _check_patches(rec, out, r, what)
    # gray, orient and line_end are views of one values tensor
    base = rec.gray.untyped_storage().data_ptr()
    assert rec.orient.untyped_storage().data_ptr() == base == rec.line_end.untyped_storage().data_ptr()
    plain = pipe.run_frames_records(frames)
    assert np.array_equal(_np(rec.frame_offsets), _np(plain.frame_offsets)), what
    _same_bits(rec.frame_yx, _np(plain.frame_yx), what + " frame_yx")
    if r == 0:   # radius 0 is the records, bit for bit
        for field in ("gray", "orient", "line_end"):
            _same_bits(_np(getattr(rec, field))[:, 0, 0], _np(getattr(plain, field)), "%s %s" % (what, field))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "float16"])
@pytest.mark.parametrize("r", (1, 3))
def test_border_patches_of_an_all_zero_level(dtype, r, cuda):
    """Every pixel of an all-zero level is a point (each equals its region maximum), so the level's corners and edges
    are: their patch pixels outside the level are +0.0 by bit pattern, those inside are the data. Rows outside the
    call's [batch * L, h, w] get NaN patches."""
    torch = cuda
    from pysilent_b200 import _ops
    plan = _geometry_plan(96, 128, (48, 32), SQRT2)
    L, h, w, b, c = plan.levels, plan.h, plan.w, 2, 4
    rs = np.random.RandomState(70 + r)
    gray = rs.uniform(0.5, 2.0, size=(b * L, h, w, 1)).astype(np.float32)
    zero = L + 1
    gray[zero] = 0
    dt = getattr(torch, dtype)
    orient = torch.from_numpy(rs.normal(size=(b * L, h, w, c)).astype(np.float32)).to("cuda", dt)
    line_end = torch.from_numpy(rs.normal(size=(b * L, h, w, c)).astype(np.float32)).to("cuda", dt)
    gray_dev = torch.from_numpy(gray).cuda()
    emitted = _np(_ops.max_value_indices_region(gray_dev, h // 2, w // 2))
    assert (emitted[:, 0] == zero).sum() == h * w
    images = b * L
    outside = np.array([[images - 1, h, 3, 0], [images - 1, 2, -1, 0], [images - 1, 2, w, 0], [images, 0, 0, 0]])
    pts = np.concatenate([emitted, outside])
    count = torch.full((1,), len(pts), dtype=torch.int64, device="cuda")
    offs, yx, vals = _ops.point_records(plan, b, torch.from_numpy(pts).cuda(), count, orient, line_end, gray_dev,
                                        radius=r)
    vals = _np(vals)
    k = len(emitted)
    want = np.concatenate([zero_padded_patches(gray[..., 0], emitted, r)[..., None],
                           zero_padded_patches(_np(orient.float()), emitted, r),
                           zero_padded_patches(_np(line_end.float()), emitted, r)], axis=-1)
    _same_bits(vals[:k], want, "%s r=%d" % (dtype, r))
    assert np.isnan(vals[k:]).all() and np.isnan(_np(yx)[k:]).all(), "rows outside the call"
    assert list(_np(offs)) == [int(np.searchsorted(pts[:, 0], f * L)) for f in range(b + 1)]
    d = np.arange(-r, r + 1)
    for y, x in ((0, 0), (0, w - 1), (h - 1, 0), (h - 1, w - 1), (0, w // 2), (h // 2, w - 1)):
        i = int(np.nonzero((emitted[:, 0] == zero) & (emitted[:, 1] == y) & (emitted[:, 2] == x))[0][0])
        out_of_level = ~(((y + d >= 0) & (y + d < h))[:, None] & ((x + d >= 0) & (x + d < w))[None, :])
        assert out_of_level.any()
        assert (vals[i][out_of_level].view(np.uint32) == 0).all(), (y, x)
        assert (vals[i][~out_of_level][:, 1:] != 0).all(), (y, x)   # the data, nonzero inside the level


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [{}, dict(orientations=8, out_dtype="f16")], ids=["f32", "bank8_f16"])
def test_capacity_contract(kw, cuda):
    torch = cuda
    size, zoom, r = (96, 64), 1.3, 2
    p = 2 * r + 1
    frames = torch.from_numpy(_bgr([("periodic", 12, 1), ("noise", 12, 0), ("struct", 3)], 480, 640)).cuda()
    pipe = _pipe(torch, size, zoom, kw)
    full = pipe.run_frames_records(frames, patch_radius=r)
    pts, offsets = _np(full.points), _np(full.frame_offsets)
    total = len(pts)
    caps = _capacities(pts, offsets)
    assert 1 < caps["in_run"] < total - 1 and 1 < caps["frame_edge"] < total - 1, caps
    c = full.orient.shape[-1]
    vals = np.concatenate([_np(full.gray)[..., None], _np(full.orient), _np(full.line_end)], axis=-1)
    L = pipe.plan_for(frames).levels
    orient = torch.empty((3 * L, size[1], size[0], c), dtype=pipe.out_dtype, device="cuda")
    line_end = torch.empty_like(orient)
    for kind, cap in caps.items():
        big_pts = torch.full((total + 16, 4), SENTINEL, dtype=torch.int64, device="cuda")
        big_yx = torch.full((total + 16, 2), FSENTINEL, dtype=torch.float32, device="cuda")
        big_val = torch.full((total + 16, p, p, 1 + 2 * c), FSENTINEL, dtype=torch.float32, device="cuda")
        offs = torch.full((4,), SENTINEL, dtype=torch.int64, device="cuda")
        count = torch.full((1,), -1, dtype=torch.int64, device="cuda")
        rec = pipe.run_frames_records(frames, out=(orient, line_end, big_pts[:cap], count, offs, big_yx[:cap],
                                                   big_val[:cap]), patch_radius=r)
        torch.cuda.synchronize()
        what = "%s cap %s=%d" % (kw, kind, cap)
        assert int(count.item()) == total, what
        assert rec.points.shape[0] == cap and tuple(rec.gray.shape) == (cap, p, p), what
        assert np.array_equal(_np(big_pts)[:cap], pts[:cap]), what
        _same_bits(_np(big_yx)[:cap], _np(full.frame_yx)[:cap], what + " frame_yx")
        _same_bits(_np(big_val)[:cap], vals[:cap], what + " values")
        assert (_np(big_pts)[cap:] == SENTINEL).all(), what + ": points past the capacity"
        assert (_np(big_yx)[cap:] == FSENTINEL).all() and (_np(big_val)[cap:] == FSENTINEL).all(), \
            what + ": patches past the capacity"
        assert np.array_equal(_np(offs), np.minimum(offsets, cap)), what + " frame_offsets"


@pytest.mark.gpu
def test_out_buffers_take_no_host_synchronisation(cuda):
    torch = cuda
    size, zoom, r = (96, 64), 1.5, 2
    pipe = _pipe(torch, size, zoom, {})
    frames = torch.from_numpy(_bgr([("noise", 60, i) for i in range(3)], 240, 320)).cuda()
    L = pipe.plan_for(frames).levels
    cap = 512
    out = (torch.empty((3 * L, 64, 96, 3), device="cuda"), torch.empty((3 * L, 64, 96, 3), device="cuda"),
           torch.empty((cap, 4), dtype=torch.int64, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda"),
           torch.empty(4, dtype=torch.int64, device="cuda"), torch.empty((cap, 2), device="cuda"),
           torch.empty((cap, 5, 5, 7), device="cuda"))
    pipe.run_frames_records(frames, out=out, patch_radius=r)   # plan set-up and workspace outside the checked call
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        rec = pipe.run_frames_records(frames, out=out, patch_radius=r)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    total = int(out[3].item())
    assert 0 < total <= cap
    want = pipe.run_frames_records(frames, patch_radius=r)
    assert np.array_equal(_np(rec.points)[:total], _np(want.points))
    _same_bits(_np(rec.orient)[:total], _np(want.orient), "orient")
    _same_bits(_np(rec.gray)[:total], _np(want.gray), "gray")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12", "bgr_f16"])
def test_host_patches_equal_device_patches(fmt, cuda):
    torch = cuda
    size, zoom, r = (288, 192), 1.3, 4
    if fmt == "nv12":
        frames = random_nv12(61, 480, 640, 3)
        kw = dict(frame_format="nv12")
    else:
        frames = _bgr([("noise", 62, i) for i in range(3)], 480, 640)
        kw = dict(out_dtype="f16") if fmt == "bgr_f16" else {}
    pipe = _pipe(torch, size, zoom, kw)
    dev_frames = torch.from_numpy(frames).cuda()
    want = pipe.run_frames_records(dev_frames, patch_radius=r)
    assert want.orient.shape[1:] == (9, 9, 3)
    redo = pipe.run_frames_records(dev_frames, points_capacity=8, patch_radius=r)   # redone with room for every point
    pinned = torch.empty(frames.shape, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[...] = frames
    for what, got in (("device, capacity 8", redo),
                      ("pageable", pipe.run_host_records(frames, points_capacity=8, patch_radius=r)),
                      ("pinned", pipe.run_host_records(pinned.numpy(), points_capacity=8, patch_radius=r)),
                      ("pinned, default capacity", pipe.run_host_records(pinned.numpy(), patch_radius=r))):
        for field in got._fields:
            if what != "device, capacity 8":
                assert isinstance(getattr(got, field), np.ndarray), (what, field)
            g, w = _np(getattr(got, field)), _np(getattr(want, field))
            if g.dtype == np.float32:
                _same_bits(g, w, "%s %s %s" % (fmt, what, field))
            else:
                assert np.array_equal(g, w), (fmt, what, field)
