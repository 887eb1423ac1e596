"""float16 outputs (``out_dtype=torch.float16``): orient and padded_line_end stored as binary16 by the fused stacks.

The rule on every entry point: each output is the float32 call's value rounded once to nearest even, which is what
``.half()`` does to it; gray and the feature points are the float32 call's, bit for bit.

CPU: the five ``_f16`` symbols, their host-side checks (which return before any CUDA call) and the ``out_dtype``
validation. GPU: bit patterns against the float32 call's ``.half()`` (identical NaN masks), and against the C oracle's
float32 ``.astype(np.float16)``.
"""
import ctypes

import numpy as np
import pytest

from conftest import structured_frame, synthetic_frame
from pysilent_b200 import _lib

torch = pytest.importorskip("torch")

SQRT2 = 2 ** .5
F16_SYMBOLS = ("silent_stack_fused_f16", "silent_stack_bank_f16", "silent_pipeline_run_f16",
               "silent_pipeline_run_orientations_f16", "silent_pipeline_run_host_f16")


def _stack_weights():
    from pysilent_b200 import LineEndPipeline
    return LineEndPipeline().stack_weights()


def _bank(n):
    from pysilent_b200.pipeline import orientation_bank_filters
    f = orientation_bank_filters(n)
    return _lib.make_orientation_bank(f["rgc"], f["rgby"], f["stripe"], f["blur"], f["end"])


def _plan(L):
    p = _lib.SilentParams(480, 640, 3, 3, 96, 64, SQRT2, _lib.SILENT_U8, 0)
    plan = ctypes.c_void_p()
    assert L.silent_plan_create(ctypes.byref(p), ctypes.byref(plan)) == 0
    return plan


# ---- CPU ------------------------------------------------------------------------------------------------------------------

def test_f16_symbols_exported_and_bound(built_lib):
    for name in F16_SYMBOLS:
        assert name in _lib.SYMBOLS, name
        fn = getattr(built_lib, name)
        assert fn.restype is ctypes.c_int and fn.argtypes, name
        base = getattr(built_lib, name[:-len("_f16")])
        assert len(fn.argtypes) == len(base.argtypes), name


def test_f16_checks_run_before_any_cuda_call(built_lib):
    """Status codes of the host-side checks. Without a GPU, a check that ran after a CUDA call would report
    SILENT_E_CUDA (-4) instead."""
    L = built_lib
    fake = ctypes.c_void_p(256)
    w = _stack_weights()
    # silent_stack_fused_f16: null pyramid, non-positive sizes, workspace too small, unstructured weights
    assert L.silent_stack_fused_f16(None, 1, 4, 4, ctypes.byref(w), None, None, None, fake, 1 << 20, None) == -1
    assert L.silent_stack_fused_f16(fake, 0, 4, 4, ctypes.byref(w), None, None, None, fake, 1 << 20, None) == -1
    assert L.silent_stack_fused_f16(fake, 1, 4, -4, ctypes.byref(w), None, None, None, fake, 1 << 20, None) == -1
    assert L.silent_stack_fused_f16(fake, 2, 4, 4, ctypes.byref(w), None, None, None, None, 0, None) == -3
    from pysilent_b200 import LineEndPipeline
    f = LineEndPipeline().filters()
    blur = f["blur"].copy()
    blur[3, 3, 1, 2] *= 2
    bad = _lib.make_stack_weights(f["rgc"], f["rgby"], f["stripe"], blur, f["end"])
    assert L.silent_stack_fused_f16(fake, 1, 4, 4, ctypes.byref(bad), None, None, None, fake, 1 << 20, None) == -5
    assert b"blur filter slices differ" in L.silent_last_error()
    assert L.silent_stack_fused_f16(fake, 0, 4, 4, ctypes.byref(w), None, None, None, fake, 1 << 20, None) == -1
    assert b"silent_stack_fused_f16" in L.silent_last_error()
    # silent_stack_bank_f16: width, structure, null pyramid, sizes
    six = _bank(16)
    six.orientations = 6
    assert L.silent_stack_bank_f16(fake, 2, 8, 8, ctypes.byref(six), None, None, None, fake, 1 << 20, None) == -2
    assert b"4, 8, 12 or 16" in L.silent_last_error()
    from pysilent_b200.pipeline import orientation_bank_filters
    f12 = orientation_bank_filters(12)
    coupled = f12["end"].copy()
    coupled[1, 1, 3, 5] = .5
    unstructured = _lib.make_orientation_bank(f12["rgc"], f12["rgby"], f12["stripe"], f12["blur"], coupled)
    assert L.silent_stack_bank_f16(fake, 2, 8, 8, ctypes.byref(unstructured), None, None, None, fake, 1 << 20, None) == -5
    b12 = _bank(12)
    assert L.silent_stack_bank_f16(None, 2, 8, 8, ctypes.byref(b12), None, None, None, fake, 1 << 20, None) == -1
    assert L.silent_stack_bank_f16(fake, 2, 0, 8, ctypes.byref(b12), None, None, None, fake, 1 << 20, None) == -1
    # pipeline entries: null arguments, batch <= 0, width, structure, capacity < 0
    plan = _plan(L)
    try:
        assert L.silent_pipeline_run_f16(None, ctypes.byref(w), fake, 1, None, None, None, None, 0, None, None) == -1
        assert L.silent_pipeline_run_f16(plan, ctypes.byref(w), None, 1, None, None, None, None, 0, None, None) == -1
        assert L.silent_pipeline_run_f16(plan, ctypes.byref(w), fake, 0, None, None, None, None, 0, None, None) == -1
        assert L.silent_pipeline_run_orientations_f16(plan, ctypes.byref(six), fake, 1, None, None, None, 0, None,
                                                      None) == -2
        assert L.silent_pipeline_run_orientations_f16(plan, ctypes.byref(unstructured), fake, 1, None, None, None, 0,
                                                      None, None) == -5
        assert L.silent_pipeline_run_orientations_f16(plan, ctypes.byref(b12), fake, -1, None, None, None, 0, None,
                                                      None) == -1
        assert L.silent_pipeline_run_host_f16(plan, ctypes.byref(w), None, 1, None, None, None, 0, None, None) == -1
        assert L.silent_pipeline_run_host_f16(plan, ctypes.byref(w), fake, 0, None, None, None, 0, None, None) == -1
        assert L.silent_pipeline_run_host_f16(plan, ctypes.byref(w), fake, 1, None, None, None, -1, None, None) == -1
        assert b"capacity" in L.silent_last_error()
    finally:
        L.silent_plan_destroy(plan)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float64, torch.int16, "float16"])
def test_out_dtype_validation(dtype):
    from pysilent_b200 import LineEndPipeline
    with pytest.raises(ValueError, match="out_dtype"):
        LineEndPipeline(out_dtype=dtype)
    for ok in (torch.float32, torch.float16):
        assert LineEndPipeline(out_dtype=ok).out_dtype == ok


def test_displayer_rejects_float16_outputs():
    from pysilent_b200.recognition_testing import LineEndDisplayer
    with pytest.raises(ValueError, match="float32"):
        LineEndDisplayer(out_dtype=torch.float16)
    LineEndDisplayer(out_dtype=torch.float32)


# ---- GPU ------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cuda(built_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert built_lib.silent_device_count() >= 1
    return torch


def _numpy(t):
    return t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def assert_half_bits(got, want, what):
    """``got`` (float16) has the bit patterns of ``want`` (float16: the float32 result rounded once), NaN masks equal."""
    g, w = _numpy(got), _numpy(want)
    assert g.dtype == np.float16 and w.dtype == np.float16, (what, g.dtype, w.dtype)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    nan_g, nan_w = np.isnan(g), np.isnan(w)
    assert np.array_equal(nan_g, nan_w), "%s: NaN masks differ (%d vs %d)" % (what, nan_g.sum(), nan_w.sum())
    same = g.view(np.uint16) == w.view(np.uint16)
    assert (same | nan_w).all(), "%s: %d of %d values differ" % (what, (~(same | nan_w)).sum(), same.size)


def check_half_of(res16, res32, what):
    """res16 (out_dtype float16) against res32 (the float32 call): outputs rounded once, gray and points identical."""
    assert_half_bits(res16.orient, res32.orient.half() if isinstance(res32.orient, torch.Tensor)
                     else res32.orient.astype(np.float16), what + " orient")
    assert_half_bits(res16.padded_line_end, res32.padded_line_end.half() if isinstance(res32.padded_line_end, torch.Tensor)
                     else res32.padded_line_end.astype(np.float16), what + " padded_line_end")
    if res32.gray is not None:
        assert res16.gray.dtype == torch.float32 and torch.equal(res16.gray.nan_to_num(-1.0), res32.gray.nan_to_num(-1.0))
    if res32.points is None:
        assert res16.points is None
    else:
        assert np.array_equal(_numpy(res16.points), _numpy(res32.points)), what + " points"


def _pipes(**kw):
    from pysilent_b200 import LineEndPipeline
    return LineEndPipeline(out_dtype=torch.float16, **kw), LineEndPipeline(**kw)


# level widths by route of a staged half tile: 96 (tile stores: w % 48 == 0), 72 (bulk rows: w % 8 == 0, not a whole
# number of 48-wide tiles), 100 and 76 (element-wise: w * 3 * 2 % 16 != 0, where float32 rows would still go by bulk copy)
ROUTES = [((240, 320), (96, 64), 1.5, 3), ((240, 320), (72, 48), 1.3, 2), ((300, 420), (100, 66), 1.4, 3),
          ((200, 304), (76, 52), 1.5, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,center,scale,batch", ROUTES)
def test_run_frames_is_the_float32_result_rounded(shape, center, scale, batch, cuda):
    """Every store route in halves, odd batches, structured frames (NaN, flagged tiles for the fix-up pass) and noise."""
    p16, p32 = _pipes(output_size=center, zoom_ratio=scale)
    frames = np.stack([structured_frame(70 + i, *shape) if i % 2 == 0 else synthetic_frame(11, i, *shape)
                       for i in range(batch)])
    dev = torch.from_numpy(frames).cuda()
    r16, r32 = p16.run_frames(dev), p32.run_frames(dev)
    assert r16.orient.dtype == torch.float16 and r16.padded_line_end.dtype == torch.float16
    check_half_of(r16, r32, "run_frames %s" % (center,))


@pytest.mark.gpu
def test_single_frames_and_low_contrast(cuda):
    """A single 1080p frame runs the one-wave 32-row full variant; low-contrast batches run the quick pass plus the
    fix-up pass on the tiles it flags."""
    p16, p32 = _pipes(zoom_ratio=SQRT2)
    for frame in (synthetic_frame(2, 0, 1080, 1920), structured_frame(5, 1080, 1920)):
        dev = torch.from_numpy(frame[None]).cuda()
        check_half_of(p16.run_frames(dev), p32.run_frames(dev), "single frame")
    p16, p32 = _pipes(zoom_ratio=1.3)
    for levels_of_grey in (2, 5, 20):
        rs = np.random.RandomState(600 + levels_of_grey)
        frames = rs.randint(0, levels_of_grey, size=(3, 480, 640, 3)).astype(np.uint8)
        frames[1, 100:300, 200:500] = 1
        dev = torch.from_numpy(frames).cuda()
        check_half_of(p16.run_frames(dev), p32.run_frames(dev), "low contrast %d" % levels_of_grey)


@pytest.mark.gpu
def test_against_the_c_oracle(cuda, c_oracle, default_filters):
    """float16 outputs equal the oracle's float32 outputs cast with astype(np.float16), for each stack kind."""
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([structured_frame(81, 240, 320), synthetic_frame(12, 1, 240, 320), structured_frame(82, 240, 320)])
    pyr = c_oracle.from_image(frames, 3, (96, 64), 1.5)
    ref = c_oracle.line_end_stack(pyr, default_filters)
    res = LineEndPipeline(output_size=(96, 64), zoom_ratio=1.5, out_dtype=torch.float16).run_frames(
        torch.from_numpy(frames).cuda())
    assert_half_bits(res.orient, ref["orient"].astype(np.float16), "oracle orient")
    assert_half_bits(res.padded_line_end, ref["padded"].astype(np.float16), "oracle padded_line_end")
    assert np.array_equal(res.points.cpu().numpy(), ref["points"])
    for n in (8, 16):
        pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=1.5, orientations=n, out_dtype=torch.float16)
        ref = c_oracle.bank_stack(pyr, pipe.bank_filters(), (32, 48), order="fused")
        res = pipe.run_frames(torch.from_numpy(frames).cuda())
        assert_half_bits(res.orient, ref["orient"].astype(np.float16), "oracle bank %d orient" % n)
        assert_half_bits(res.padded_line_end, ref["padded"].astype(np.float16), "oracle bank %d padded_line_end" % n)
        assert np.array_equal(res.points.cpu().numpy(), ref["points"]), n


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 8, 12, 16])
def test_bank_run_frames(n, cuda):
    for shape, center, scale, batch in (((240, 320), (96, 64), 1.5, 3), ((200, 304), (76, 52), 1.5, 2),
                                        ((120, 160), (72, 48), 1.3, 1)):
        p16, p32 = _pipes(output_size=center, zoom_ratio=scale, orientations=n)
        frames = np.stack([structured_frame(30 + i, *shape) if i % 2 else synthetic_frame(13, i, *shape)
                           for i in range(batch)])
        dev = torch.from_numpy(frames).cuda()
        r16 = p16.run_frames(dev)
        assert r16.orient.shape[-1] == n
        check_half_of(r16, p32.run_frames(dev), "bank %d %s" % (n, center))


@pytest.mark.gpu
def test_bank_pyramids_and_operator_path(cuda):
    """run(pyramid) at 12 and 16 orientations goes through silent_stack_bank_f16 (level widths for each route, odd
    widths element-wise); 8 orientations on float frames go operator by operator and cast once."""
    rs = np.random.RandomState(21)
    for n in (12, 16):
        p16, p32 = _pipes(output_size=(96, 64), orientations=n)
        for h, w in ((64, 96), (37, 53), (40, 72)):
            pyr = (rs.rand(3, h, w, 3) * 255).astype(np.float32)
            pyr[0, : h // 3, : w // 2] = 37.0
            pyr[-1, h // 2:, w // 2:] = 0.0
            check_half_of(p16.run(pyr), p32.run(pyr), "bank %d pyramid %dx%d" % (n, h, w))
    p16, p32 = _pipes(output_size=(96, 64), zoom_ratio=1.5, orientations=8)
    frames = torch.from_numpy(np.stack([synthetic_frame(14, i, 240, 320) for i in range(2)]).astype(np.float32)).cuda()
    check_half_of(p16.run_frames(frames), p32.run_frames(frames), "bank 8, float frames")


@pytest.mark.gpu
def test_run_on_pyramids(cuda):
    """The three-orientation stack on finite pyramids (silent_stack_fused_f16) and on non-finite ones (operator by
    operator, then one cast)."""
    rs = np.random.RandomState(22)
    p16, p32 = _pipes(output_size=(96, 64))
    for n, h, w in ((2, 64, 96), (1, 37, 53), (3, 40, 100), (2, 48, 72)):
        pyr = (rs.rand(n, h, w, 3) * 255).astype(np.float32)
        pyr[0, : h // 3, : w // 2] = 37.0
        pyr[-1, h // 2:, w // 2:] = 0.0
        check_half_of(p16.run(pyr), p32.run(pyr), "pyramid %s" % ((n, h, w),))
        pyr[0, 5, 7, 1] = np.nan
        pyr[-1, 2, 3, 0] = np.inf
        check_half_of(p16.run(pyr), p32.run(pyr), "non-finite pyramid %s" % ((n, h, w),))
        check_half_of(p16.run_unfused(pyr), p32.run_unfused(pyr), "run_unfused %s" % ((n, h, w),))


@pytest.mark.gpu
def test_run_host_and_callback(cuda):
    p16, p32 = _pipes(output_size=(100, 66), zoom_ratio=1.4)
    frames = np.stack([structured_frame(91, 300, 420), synthetic_frame(15, 1, 300, 420), structured_frame(92, 300, 420)])
    r32 = p32.run_host(frames)
    pageable = p16.run_host(frames)
    assert pageable.orient.dtype == np.float16
    check_half_of(pageable, r32, "run_host pageable")
    pinned = torch.from_numpy(frames).pin_memory().numpy()
    check_half_of(p16.run_host(pinned), r32, "run_host pinned")
    orient_out = np.full(r32.orient.shape, 7, np.float16)
    line_end_out = torch.empty(r32.orient.shape, dtype=torch.float16).pin_memory().numpy()
    res = p16.run_host(frames, orient_out=orient_out, line_end_out=line_end_out)
    assert res.orient is orient_out and res.padded_line_end is line_end_out
    check_half_of(res, r32, "run_host caller buffers")
    with pytest.raises(ValueError, match="np.float16"):
        p16.run_host(frames, orient_out=np.empty(r32.orient.shape, np.float32))
    # the float32 call after a float16 one on the same plan (pinned mirrors sized per element type) is unchanged
    again = p32.run_host(frames)
    assert np.array_equal(again.orient, r32.orient, equal_nan=True) and np.array_equal(again.points, r32.points)
    cb16, cb32 = p16.callback(frames[0]), p32.callback(frames[0])
    assert len(cb16) == 4 and len(cb16[1]) == len(cb32[1]) and len(cb16[2]) == len(cb32[2])
    for a, b in zip(cb16[1] + cb16[2], cb32[1] + cb32[2]):
        assert a.dtype == np.float16 and a.shape == b.shape
        assert_half_bits(a, b.astype(np.float16), "callback level")
    assert np.array_equal(cb16[3], cb32[3])
    for n in (8, 12):
        b16, b32 = _pipes(output_size=(96, 64), zoom_ratio=1.5, orientations=n)
        check_half_of(b16.run_host(frames[:, :240, :320]), b32.run_host(frames[:, :240, :320]), "run_host bank %d" % n)


@pytest.mark.gpu
def test_out_buffers_filled_in_place(cuda):
    for n in (None, 16):
        p16, p32 = _pipes(output_size=(96, 64), zoom_ratio=1.5, orientations=n)
        dev = torch.from_numpy(np.stack([synthetic_frame(16, i, 240, 320) for i in range(3)])).cuda()
        want = p32.run_frames(dev)
        orient = torch.empty(want.orient.shape, dtype=torch.float16, device="cuda")
        line_end = torch.empty_like(orient)
        points = torch.empty((4096, 4), dtype=torch.int64, device="cuda")
        count = torch.zeros(1, dtype=torch.int64, device="cuda")
        res = p16.run_frames(dev, out=(orient, line_end, points, count))
        assert res.orient is orient and res.padded_line_end is line_end
        check_half_of(type(want)(orient, line_end, None, points[: int(count.item())]), want, "out= %s" % n)
        with pytest.raises(ValueError, match="float16"):
            p16.run_frames(dev, out=(orient.float(), line_end, points, count))
        with pytest.raises(ValueError, match="float32"):
            p32.run_frames(dev, out=(orient, line_end, points, count))


@pytest.mark.gpu
def test_half_outputs_stay_inside_their_buffers(cuda):
    """Canaries around float16 outputs: full tiles, ragged tiles, an odd batch, and level widths whose route depends on
    the element size (100 and 76: element-wise in halves, bulk rows in floats; 72: bulk rows; 96, 288: tile stores)."""
    from pysilent_b200 import LineEndPipeline
    guard = 4096   # int64 words = 32 KB between tensors
    for (shape, center, scale, batch, n_or) in (((300, 420), (100, 66), 2 ** .5, 3, None),
                                                ((200, 304), (76, 52), 1.5, 2, None),
                                                ((240, 330), (72, 48), 1.4, 3, None),
                                                ((1080, 1920), (288, 192), 2 ** .5, 5, None),
                                                ((240, 320), (96, 64), 1.5, 3, 4), ((200, 304), (76, 52), 1.5, 3, 12)):
        frames = np.stack([synthetic_frame(17, i, *shape) for i in range(batch)])
        pipe = LineEndPipeline(output_size=center, zoom_ratio=scale, orientations=n_or, out_dtype=torch.float16)
        dev = torch.from_numpy(frames).cuda()
        plan = pipe.plan_for(dev)
        n = batch * plan.levels
        ch = n_or or 3
        elems = n * plan.h * plan.w * ch
        words_t = (elems * 2 + 7) // 8
        cap = 64 * n
        arena = torch.full((5 * guard + 2 * words_t + cap * 4 + 1,), 0x5A5A5A5A5A5A5A5A, dtype=torch.int64, device="cuda")
        off = guard
        orient = arena[off: off + words_t].view(torch.float16)[:elems].view(n, plan.h, plan.w, ch)
        off += words_t + guard
        line_end = arena[off: off + words_t].view(torch.float16)[:elems].view(n, plan.h, plan.w, ch)
        off += words_t + guard
        points = arena[off: off + cap * 4].view(cap, 4)
        off += cap * 4 + guard
        count = arena[off: off + 1]
        count.zero_()
        used = torch.zeros_like(arena, dtype=torch.bool)
        for t in (orient, line_end, points, count):
            start = (t.data_ptr() - arena.data_ptr()) // 8
            used[start: start + (t.numel() * t.element_size() + 7) // 8] = True
        pipe.run_frames(dev, out=(orient, line_end, points, count))
        torch.cuda.synchronize()
        assert bool((arena[~used] == 0x5A5A5A5A5A5A5A5A).all()), "a kernel wrote outside its outputs %s" % (center,)
        ref = pipe.run_frames(dev)
        assert torch.equal(ref.orient.view(torch.int16), orient.view(torch.int16))
        assert torch.equal(ref.padded_line_end.view(torch.int16), line_end.view(torch.int16))
        assert torch.equal(ref.points, points[: int(count.item())])
