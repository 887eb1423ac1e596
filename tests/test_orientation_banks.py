"""Orientation banks of 4, 8, 12 and 16 orientations (config C4 and its variants) through every entry point.

CPU: the C struct's layout, the packing helper, the generators' structure and every width / structure check (which run
before anything touches the GPU). GPU: the fused bank paths against the bit-defined C oracle (values, NaN masks and
point rows bitwise), as for the 8-orientation bank in test_gpu_parity.py.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, structured_frame, synthetic_frame
from pysilent_b200 import _lib

SQRT2 = 2 ** .5


def _filters(n):
    from pysilent_b200.pipeline import orientation_bank_filters
    return orientation_bank_filters(n)


def _bank(f, **kw):
    return _lib.make_orientation_bank(f["rgc"], f["rgby"], f["stripe"], f["blur"], f["end"], **kw)


# ---- CPU ------------------------------------------------------------------------------------------------------------------

def test_struct_layout_matches_the_header(tmp_path):
    fields = [name for name, _ in _lib.SilentOrientationBank._fields_]
    src = tmp_path / "probe.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "silent_b200.h"\nint main(void){\n'
                   '  printf("sizeof %zu\\n", sizeof(silent_orientation_bank));\n'
                   + "".join('  printf("%s %%zu %%zu\\n", offsetof(silent_orientation_bank, %s), '
                             'sizeof(((silent_orientation_bank *)0)->%s));\n' % (f, f, f) for f in fields)
                   + '  printf("max %d\\n", SILENT_BANK_MAX);\n  return 0;\n}\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o",
                           str(exe)])
    out = dict((line.split()[0], line.split()[1:]) for line in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(out["sizeof"][0]) == ctypes.sizeof(_lib.SilentOrientationBank)
    assert int(out["max"][0]) == _lib.BANK_MAX
    for f in fields:
        desc = getattr(_lib.SilentOrientationBank, f)
        assert [int(v) for v in out[f]] == [desc.offset, desc.size], f


def test_make_orientation_bank_shapes_and_packing():
    f8 = _filters(8)
    b = _bank(f8)
    w = _lib.make_bank_weights(f8["rgc"], f8["rgby"], f8["stripe"], f8["blur"], f8["end"])
    assert b.orientations == 8
    for name in ("rgc", "rgby", "stripe", "blur", "end"):
        assert bytes(getattr(w, name)) == bytes(getattr(b, name))[:ctypes.sizeof(getattr(w, name))], name
    assert (b.regulation_value, b.regulation_root, b.clip_max, b.border) == \
        (w.regulation_value, w.regulation_root, w.clip_max, w.border)
    f12 = _filters(12)
    b12 = _bank(f12)
    assert b12.orientations == 12
    assert np.array_equal(np.frombuffer(b12.blur, np.float32)[:49 * 144], f12["blur"].astype(np.float32).ravel())
    assert not np.frombuffer(b12.blur, np.float32)[49 * 144:].any()
    bad = [dict(stripe=f8["stripe"][:, :, :, :0]), dict(stripe=np.zeros((3, 3, 3, 17))), dict(stripe=f8["stripe"][:2]),
           dict(blur=f12["blur"]), dict(end=f12["end"]), dict(blur=f8["blur"][:5, :5]), dict(rgc=f8["rgc"][:, :, :2])]
    for change in bad:
        g = dict(f8, **change)
        with pytest.raises(ValueError):
            _bank(g)


@pytest.mark.parametrize("n", [4, 12, 16])
def test_generators_give_the_structure_the_bank_kernel_needs(n):
    f = {k: np.asarray(v, np.float32) for k, v in _filters(n).items()}
    assert f["stripe"].shape == (3, 3, 3, n) and f["blur"].shape == (7, 7, n, n) and f["end"].shape == (3, 3, n, n)
    assert (f["stripe"] == f["stripe"][:, :, :1, :]).all()                         # identical over the input channels
    assert (f["blur"] == f["blur"][:, :, :1, :1]).all()                            # every slice identical
    off = ~np.eye(n, dtype=bool)
    assert not f["end"][:, :, off].any() and f["end"][:, :, ~off].any()            # depthwise


def _host_checks(L, bank):
    """(silent_stack_bank, silent_pipeline_run_orientations) status on fake device pointers: only the host-side checks
    can return before a CUDA call."""
    p = _lib.SilentParams(480, 640, 3, 3, 96, 64, SQRT2, _lib.SILENT_U8, 0)
    plan = ctypes.c_void_p()
    assert L.silent_plan_create(ctypes.byref(p), ctypes.byref(plan)) == 0
    try:
        rc_stack = L.silent_stack_bank(ctypes.c_void_p(256), 2, 8, 8, ctypes.byref(bank), None, None, None,
                                       ctypes.c_void_p(256), 1 << 20, None)
        msg_stack = L.silent_last_error()
        rc_pipe = L.silent_pipeline_run_orientations(plan, ctypes.byref(bank), ctypes.c_void_p(256), 1, None, None, None,
                                                     0, None, None)
        msg_pipe = L.silent_last_error()
    finally:
        L.silent_plan_destroy(plan)
    return (rc_stack, msg_stack), (rc_pipe, msg_pipe)


def test_width_and_structure_checks_are_host_side(built_lib):
    for n in (6, 20):
        bank = _bank(_filters(6)) if n == 6 else _bank(_filters(16))
        bank.orientations = n
        for rc, msg in _host_checks(built_lib, bank):
            assert rc == -2 and b"4, 8, 12 or 16" in msg, (n, rc, msg)
    f = _filters(12)
    coupled = f["end"].copy()
    coupled[1, 1, 3, 5] = .5
    stripe = f["stripe"].copy()
    stripe[0, 2, 1, 7] += 1.0
    blur = f["blur"].copy()
    blur[3, 3, 11, 2] *= 2
    for change, text in ((dict(end=coupled), b"end bank couples orientations 3 -> 5"),
                         (dict(stripe=stripe), b"stripe bank differs across input channels at tap 2"),
                         (dict(blur=blur), b"blur bank slices differ at tap 24")):
        for rc, msg in _host_checks(built_lib, _bank(dict(f, **change))):
            assert rc == -5 and text in msg, (rc, msg)


@pytest.mark.parametrize("n", [9, 10, 14, 20, 32])
def test_unsupported_widths_fail_before_the_gpu(n):
    """Each entry point rejects the width before anything touches CUDA (these inputs are CPU tensors / numpy arrays, so
    a later check would fail differently, and on a machine without a GPU with RuntimeError)."""
    torch = pytest.importorskip("torch")
    from pysilent_b200 import LineEndPipeline
    from pysilent_b200.recognition_testing import LineEndDisplayer
    frame = np.zeros((240, 320, 3), np.uint8)
    pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=SQRT2, orientations=n)
    calls = [lambda: pipe.run_frames(torch.from_numpy(frame[None])), lambda: pipe.run(np.zeros((2, 64, 96, 3), np.float32)),
             lambda: pipe.run_bank(np.zeros((2, 64, 96, 3), np.float32)), lambda: pipe.run_host(frame),
             lambda: pipe.callback(frame), lambda: LineEndDisplayer(orientations=n).callback(frame)]
    for call in calls:
        with pytest.raises(ValueError, match="12 or 16"):
            call()


# ---- GPU ------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cuda(built_lib):
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert built_lib.silent_device_count() >= 1
    return torch


def assert_bits(actual, expected, what):
    a = actual.detach().cpu().numpy() if hasattr(actual, "detach") else np.asarray(actual)
    e = np.asarray(expected)
    assert a.shape == e.shape, (what, a.shape, e.shape)
    nan_a, nan_e = np.isnan(a), np.isnan(e)
    assert np.array_equal(nan_a, nan_e), "%s: NaN masks differ (%d vs %d)" % (what, nan_a.sum(), nan_e.sum())
    same = (a == e) | nan_e
    assert same.all(), "%s: %d of %d values differ from the bit-defined oracle" % (what, (~same).sum(), same.size)


def check_against(res, ref, what):
    assert_bits(res.orient, ref["orient"], what + " orient")
    assert_bits(res.padded_line_end, ref["padded"], what + " padded_line_end")
    if res.gray is not None:
        assert_bits(res.gray, ref["gray"], what + " gray")
    pts = res.points.cpu().numpy() if hasattr(res.points, "cpu") else res.points
    assert np.array_equal(pts, ref["points"]), what + " points"


def _oracle(c_oracle, frames, pipe, center, scale):
    pyr = c_oracle.from_image(frames, 3, center, scale)
    return pyr, c_oracle.bank_stack(pyr, pipe.bank_filters(), (center[1] // 2, center[0] // 2), order="fused")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 12, 16])
def test_bank_run_frames_bit_exact(n, cuda, c_oracle):
    """Fused bank path at widths 4, 12, 16: structured frames (regulator slow path, NaN from the black patch) and noise,
    odd batch (a lone frame in the last pair); bitwise against the oracle's fused order, orient within 2e-5 of the
    literal oracle."""
    from oracle import silent_oracle as lit
    from pysilent_b200 import LineEndPipeline
    pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=SQRT2, orientations=n)
    frames = np.stack([structured_frame(170 + i, 300, 432) if i != 1 else synthetic_frame(4, i, 300, 432)
                       for i in range(3)])
    pyr, ref = _oracle(c_oracle, frames, pipe, (96, 64), SQRT2)
    res = pipe.run_frames(cuda.from_numpy(frames).cuda())
    assert tuple(res.orient.shape) == pyr.shape[:3] + (n,)
    check_against(res, ref, "bank %d" % n)
    assert np.isnan(ref["orient"]).any()
    f = pipe.bank_filters()
    lit_orient = lit.regulate_tensor(lit.conv_relu(lit.conv_relu(lit.conv_relu(pyr, f["rgc"]), f["rgby"]), f["stripe"]),
                                     f["blur"], 1.0, .1)
    a, e = res.orient.cpu().numpy(), np.asarray(lit_orient)
    assert np.array_equal(np.isnan(a), np.isnan(e))
    assert np.nanmax(np.abs(a - e)) <= 2e-5 * np.nanmax(np.abs(e))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [12, 16])
def test_bank_shape_sweep_bit_exact(n, cuda, c_oracle):
    """The cases of test_orientation_bank_shape_sweep_bit_exact at the wide banks, plus a 50-wide level (not a multiple
    of the 16- or 32-column tile, nor of 4: the bulk-row and element-wise store fallbacks)."""
    from pysilent_b200 import LineEndPipeline
    cases = [((120, 160), (72, 48), 1.3, 2), ((200, 304), (76, 52), 1.5, 3), ((333, 448), (144, 96), 1.25, 1),
             ((480, 640), (100, 66), 1.7, 3), ((96, 128), (34, 18), 1.6, 5), ((120, 176), (50, 34), 1.4, 3)]
    for shape, center, scale, batch in cases:
        frames = np.stack([structured_frame(60 + i, *shape) if i % 2 else synthetic_frame(9, i, *shape)
                           for i in range(batch)])
        pipe = LineEndPipeline(output_size=center, zoom_ratio=scale, orientations=n)
        pyr, ref = _oracle(c_oracle, frames, pipe, center, scale)
        res = pipe.run_frames(cuda.from_numpy(frames).cuda())
        assert tuple(res.orient.shape) == pyr.shape[:3] + (n,)
        check_against(res, ref, "bank %d %s" % (n, shape))


@pytest.mark.gpu
def test_bank16_at_4k(cuda, c_oracle):
    """n = 16 at C4's named shape: one 3840x2160 frame, all 8 levels, against the oracle; batch independence and
    determinism on a batch of two."""
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([synthetic_frame(4, i, 2160, 3840) for i in range(2)])
    pipe = LineEndPipeline(zoom_ratio=SQRT2, orientations=16)
    dev = cuda.from_numpy(frames).cuda()
    one = pipe.run_frames(dev[:1])
    pyr, ref = _oracle(c_oracle, frames[:1], pipe, (288, 192), SQRT2)
    assert pyr.shape == (8, 192, 288, 3)
    check_against(one, ref, "bank 16 at 4K")
    full = pipe.run_frames(dev)
    assert tuple(full.orient.shape) == (16, 192, 288, 16)
    last = pipe.run_frames(dev[1:2])
    assert cuda.equal(last.orient, full.orient[8:]) and cuda.equal(last.padded_line_end, full.padded_line_end[8:])
    again = pipe.run_frames(dev)
    assert cuda.equal(again.orient, full.orient) and cuda.equal(again.padded_line_end, full.padded_line_end)
    assert cuda.equal(again.points, full.points)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [8, 16])
def test_bank_run_frames_into_caller_buffers(n, cuda):
    """run_frames(frames, out=bufs) with orientations set fills the caller's (orient, padded_line_end, points, count), as
    for the 3-orientation stack, bit for bit what the call without out returns."""
    from pysilent_b200 import LineEndPipeline
    pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=SQRT2, orientations=n)
    frames = cuda.from_numpy(np.stack([structured_frame(90 + i, 300, 432) for i in range(3)])).cuda()
    ref = pipe.run_frames(frames)
    bufs = (cuda.full_like(ref.orient, -7.0), cuda.full_like(ref.padded_line_end, -7.0),
            cuda.full((64 * ref.orient.shape[0], 4), -1, dtype=cuda.int64, device="cuda"),
            cuda.zeros(1, dtype=cuda.int64, device="cuda"))
    res = pipe.run_frames(frames, out=bufs)
    assert res.orient is bufs[0] and res.padded_line_end is bufs[1] and res.points is bufs[2]
    assert cuda.equal(bufs[0].view(cuda.int32), ref.orient.view(cuda.int32))
    assert cuda.equal(bufs[1].view(cuda.int32), ref.padded_line_end.view(cuda.int32))
    count = int(bufs[3].item())
    assert count == ref.points.shape[0] and cuda.equal(bufs[2][:count], ref.points)


@pytest.mark.gpu
def test_bank8_new_entry_equals_old_entry(cuda):
    """At n = 8, silent_pipeline_run_orientations, silent_pipeline_run_bank and run_frames agree bit for bit."""
    from pysilent_b200 import LineEndPipeline, _ops
    pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=SQRT2, orientations=8)
    frames = cuda.from_numpy(np.stack([structured_frame(80 + i, 300, 432) for i in range(3)])).cuda()
    res = pipe.run_frames(frames)
    plan = pipe.plan_for(frames)
    n = 3 * plan.levels
    f = pipe.bank_filters()
    old = _lib.make_bank_weights(f["rgc"], f["rgby"], f["stripe"], f["blur"], f["end"])
    outs = {}
    for name, fn, weights in (("old", "silent_pipeline_run_bank", old),
                              ("new", "silent_pipeline_run_orientations", pipe.orientation_bank())):
        o = cuda.full((n, plan.h, plan.w, 8), -7.0, device="cuda")
        l = cuda.full_like(o, -7.0)
        pts = cuda.empty((64 * n, 4), dtype=cuda.int64, device="cuda")
        cnt = cuda.zeros(1, dtype=cuda.int64, device="cuda")
        _lib.check(getattr(_lib.lib(), fn)(plan.handle, ctypes.byref(weights), _ops.ptr(frames), 3, _ops.ptr(o), _ops.ptr(l),
                                           _ops.ptr(pts), 64 * n, _ops.ptr(cnt), _ops.stream_ptr()), fn)
        outs[name] = (o, l, pts[: int(cnt.item())])
    for name, (o, l, pts) in outs.items():
        assert cuda.equal(o.nan_to_num(-1.0), res.orient.nan_to_num(-1.0)), name
        assert cuda.equal(l.nan_to_num(-1.0), res.padded_line_end.nan_to_num(-1.0)), name
        assert cuda.equal(pts, res.points), name


@pytest.mark.gpu
def test_bank16_on_pyramids_and_float_frames(cuda, c_oracle):
    """silent_stack_bank through run(pyramid) on a finite NHWC pyramid (odd count: a lone image in the last pair) and
    through run_frames on float32 frames (pyramid first): bitwise against the oracle's fused order. A pyramid with a
    NaN raises ValueError."""
    from pysilent_b200 import LineEndPipeline, _ops
    pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=SQRT2, orientations=16)
    frames = np.stack([structured_frame(50 + i, 300, 432) for i in range(2)])
    pyr = c_oracle.from_image(frames, 3, (96, 64), SQRT2)[:-1]
    ref = c_oracle.bank_stack(pyr, pipe.bank_filters(), (32, 48), order="fused")
    check_against(pipe.run(pyr), ref, "run(pyramid)")
    orient, line_end, gray = _ops.stack_bank(pyr, pipe.orientation_bank())
    assert_bits(orient, ref["orient"], "stack_bank orient")
    assert_bits(line_end, ref["padded"], "stack_bank padded_line_end")
    assert_bits(gray, ref["gray"], "stack_bank gray")
    bad = pyr.copy()
    bad[1, 5, 7, 2] = np.nan
    with pytest.raises(ValueError, match="at most 8"):
        pipe.run(bad)
    ff = frames.astype(np.float32)
    pyr_f, ref_f = _oracle(c_oracle, ff, pipe, (96, 64), SQRT2)
    check_against(pipe.run_frames(cuda.from_numpy(ff).cuda()), ref_f, "float32 frames")


@pytest.mark.gpu
def test_bank16_host_entry_points(cuda):
    """run_host honours orientations (equal to run_frames bit for bit, into caller buffers too); LineEndPipeline.callback
    returns 16-channel level images; LineEndDisplayer.callback returns the six display lists."""
    from pysilent_b200 import LineEndPipeline
    from pysilent_b200.recognition_testing import LineEndDisplayer
    pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=SQRT2, orientations=16)
    frames = np.stack([structured_frame(20 + i, 300, 432) for i in range(3)])
    dev = pipe.run_frames(cuda.from_numpy(frames).cuda())
    host = pipe.run_host(frames)
    assert np.array_equal(host.orient, dev.orient.cpu().numpy(), equal_nan=True)
    assert np.array_equal(host.padded_line_end, dev.padded_line_end.cpu().numpy(), equal_nan=True)
    assert np.array_equal(host.points, dev.points.cpu().numpy())
    o, l = np.empty_like(host.orient), np.empty_like(host.padded_line_end)
    small = pipe.run_host(frames, o, l, points_capacity=1)
    assert small.orient is o and np.array_equal(o, host.orient, equal_nan=True)
    assert np.array_equal(l, host.padded_line_end, equal_nan=True) and np.array_equal(small.points, host.points)
    L = dev.orient.shape[0] // 3
    frame = frames[0]
    out = pipe.callback(frame)
    assert out[0] is frame and len(out[1]) == L and len(out[2]) == L
    assert out[1][0].shape == (64, 96, 16) and out[2][0].shape == (64, 96, 16)
    assert np.array_equal(np.stack(out[1]), host.orient[:L], equal_nan=True)
    assert np.array_equal(np.stack(out[2]), host.padded_line_end[:L], equal_nan=True)
    disp = LineEndDisplayer(output_size=(96, 64), zoom_ratio=SQRT2, orientations=16)
    shown = disp.callback(frame)
    assert shown[0] is frame and len(shown) == 7 and all(len(shown[1 + x]) == L for x in range(6))
    assert shown[1][0].shape == (64, 96, 16) and shown[6][0].shape == (64, 96, 16) and shown[2][0].shape == (64, 96, 1)
    assert np.array_equal(np.stack(shown[1]), host.orient[:L], equal_nan=True)
