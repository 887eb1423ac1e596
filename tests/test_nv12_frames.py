"""NV12 frames (``frame_format="nv12"``, ``SILENT_NV12`` plans, ``silent_nv12_to_bgr``).

The rule on every entry point: an NV12 call returns exactly what the same call returns on the BGR frames
``cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12)`` makes of them. ``nv12_to_bgr_reference`` restates that conversion in
numpy (OpenCV's integer code); a CPU test pins it to cv2 itself, and the GPU tests compare against it, so they do not
need cv2.

CPU: the restatement against cv2, the exported symbol, plan geometry, the host-side status codes (which return before
any CUDA call) and the Python validation. GPU: bit patterns and NaN masks against the same call on the reference-converted
BGR frames.
"""
import ctypes

import numpy as np
import pytest

from pysilent_b200 import _lib

torch = pytest.importorskip("torch")

SQRT2 = 2 ** .5


def nv12_to_bgr_reference(nv12):
    """cv2.cvtColor(nv12, cv2.COLOR_YUV2BGR_NV12) for ``[..., H * 3 / 2, W]`` uint8: BT.601 limited range in 20-bit
    fixed point, one (U, V) pair per 2 x 2 block."""
    nv12 = np.asarray(nv12)
    rows, w = nv12.shape[-2:]
    h = 2 * rows // 3
    y = nv12[..., :h, :].astype(np.int64)
    uv = nv12[..., h:, :].reshape(nv12.shape[:-2] + (h // 2, w // 2, 2)).astype(np.int64)
    u = np.repeat(np.repeat(uv[..., 0], 2, -2), 2, -1) - 128
    v = np.repeat(np.repeat(uv[..., 1], 2, -2), 2, -1) - 128
    yy = np.maximum(0, y - 16) * 1220542
    half = 1 << 19
    b = (yy + half + 2116026 * u) >> 20
    g = (yy + half - 852492 * v - 409993 * u) >> 20
    r = (yy + half + 1673527 * v) >> 20
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)


def random_nv12(seed, h, w, batch=None):
    rs = np.random.RandomState(seed)
    shape = (h * 3 // 2, w) if batch is None else (batch, h * 3 // 2, w)
    return rs.randint(0, 256, size=shape).astype(np.uint8)


def structured_nv12(seed, h, w):
    """Edges and smooth shading, flat patches, and a patch of Y <= 16 with neutral chroma: black BGR, which drives the
    regulator's 0 * inf = NaN path."""
    img = random_nv12(seed, h, w)
    y, uv = img[:h], img[h:].reshape(h // 2, w // 2, 2)
    yy, xx = np.mgrid[0:h, 0:w]
    y[: h // 3] = (96 + 80 * np.sin(xx / 9.0) * np.cos(yy / 7.0)).astype(np.uint8)[: h // 3]
    y0, y1, x0, x1 = (2 * h) // 5 & ~1, (3 * h) // 5 & ~1, (2 * w) // 5 & ~1, (3 * w) // 5 & ~1
    y[y0:y1, x0:x1] = np.random.RandomState(seed + 1).randint(0, 17, size=(y1 - y0, x1 - x0))
    uv[y0 // 2: y1 // 2, x0 // 2: x1 // 2] = 128
    fy0, fy1, fx0, fx1 = (7 * h) // 10 & ~1, (9 * h) // 10 & ~1, w // 10 & ~1, (4 * w) // 10 & ~1
    y[fy0:fy1, fx0:fx1] = 60
    uv[fy0 // 2: fy1 // 2, fx0 // 2: fx1 // 2] = (90, 170)
    return img


def _geometry_plan(L, H, W, dtype, c=3, nc=3, center=(96, 64), scale=SQRT2):
    p = _lib.SilentParams(H, W, c, nc, center[0], center[1], float(scale), dtype, 0)
    h = ctypes.c_void_p()
    rc = L.silent_plan_create(ctypes.byref(p), ctypes.byref(h))
    return rc, h


# ---- CPU ------------------------------------------------------------------------------------------------------------------

def test_reference_equals_cv2_on_every_triple_and_random_frames():
    cv2 = pytest.importorskip("cv2")
    u, v = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    uv = np.stack([u, v], -1).astype(np.uint8).reshape(256, 512)   # 2 x 2 block (i, j) has (U, V) = (i, j)
    for y in range(256):                                            # ... and Y = y everywhere: all 2^24 triples
        img = np.concatenate([np.full((512, 512), y, np.uint8), uv], 0)
        assert np.array_equal(nv12_to_bgr_reference(img), cv2.cvtColor(img, cv2.COLOR_YUV2BGR_NV12)), y
    for seed, (h, w) in enumerate(((1080, 1920), (480, 640), (768, 1366), (1920, 1080), (6, 10), (2, 2))):
        img = random_nv12(seed, h, w)
        want = cv2.cvtColor(img, cv2.COLOR_YUV2BGR_NV12)
        assert want.shape == (h, w, 3)
        assert np.array_equal(nv12_to_bgr_reference(img), want), (h, w)
    img = structured_nv12(3, 120, 160)
    assert np.array_equal(nv12_to_bgr_reference(img), cv2.cvtColor(img, cv2.COLOR_YUV2BGR_NV12))
    batch = random_nv12(9, 8, 6, batch=3)
    assert np.array_equal(nv12_to_bgr_reference(batch), np.stack([nv12_to_bgr_reference(f) for f in batch]))


def test_nv12_symbol_exported_and_bound(built_lib):
    assert "silent_nv12_to_bgr" in _lib.SYMBOLS
    fn = built_lib.silent_nv12_to_bgr
    assert fn.restype is ctypes.c_int and len(fn.argtypes) == 6
    assert _lib.SILENT_NV12 == 2


@pytest.mark.parametrize("H,W,center,scale", [(1080, 1920, (288, 192), SQRT2), (768, 1366, (96, 64), 1.5),
                                              (1920, 1080, (100, 66), 1.4), (482, 642, (72, 48), 1.3)])
def test_nv12_plan_geometry_is_the_bgr_plans(H, W, center, scale, built_lib):
    L = built_lib
    rc, bgr = _geometry_plan(L, H, W, _lib.SILENT_U8, center=center, scale=scale)
    assert rc == 0
    rc, nv12 = _geometry_plan(L, H, W, _lib.SILENT_NV12, center=center, scale=scale)
    assert rc == 0
    try:
        levels = L.silent_plan_levels(bgr)
        assert levels > 0 and L.silent_plan_levels(nv12) == levels
        h, w = center[1], center[0]
        union_h = union_w = 0
        for s in range(levels):
            infos = []
            for plan in (bgr, nv12):
                vals = [ctypes.c_int() for _ in range(6)]
                assert L.silent_plan_level_info(plan, s, *[ctypes.byref(v) for v in vals]) == 0
                infos.append(tuple(v.value for v in vals))
                tabs = (np.empty((h, 6), np.int32), np.empty((h, 6), np.float32), np.empty((w, 6), np.int32),
                        np.empty((w, 6), np.float32))
                assert L.silent_plan_level_tables(plan, s, *[t.ctypes.data for t in tabs]) == 0
                infos.append(b"".join(t.tobytes() for t in tabs))
            assert infos[0] == infos[2] and infos[1] == infos[3], s
            y0, y1, x0, x1 = infos[0][:4]
            union_h, union_w = max(union_h, y1 - y0), max(union_w, x1 - x0)
        out_bytes = 2 * levels * h * w * 3 * 4
        assert L.silent_plan_algorithmic_bytes(bgr) == union_h * union_w * 3 + out_bytes
        assert L.silent_plan_algorithmic_bytes(nv12) == union_h * union_w * 3 // 2 + out_bytes
    finally:
        L.silent_plan_destroy(bgr)
        L.silent_plan_destroy(nv12)


def test_nv12_checks_run_before_any_cuda_call(built_lib):
    """Status codes of the host-side checks. Without a GPU, a check that ran after a CUDA call would report
    SILENT_E_CUDA (-4) instead."""
    L = built_lib
    for H, W in ((481, 640), (480, 641), (3, 3)):
        assert _geometry_plan(L, H, W, _lib.SILENT_NV12)[0] == -2, (H, W)
        assert b"even" in L.silent_last_error()
    assert _geometry_plan(L, 480, 640, _lib.SILENT_NV12, c=4, nc=3)[0] == -2
    assert _geometry_plan(L, 480, 640, _lib.SILENT_NV12, c=3, nc=2)[0] == -2
    assert b"num_colors" in L.silent_last_error()
    assert _geometry_plan(L, 480, 640, 3)[0] == -1
    fake = ctypes.c_void_p(256)
    assert L.silent_nv12_to_bgr(None, 1, 4, 4, fake, None) == -1
    assert L.silent_nv12_to_bgr(fake, 1, 4, 4, None, None) == -1
    assert L.silent_nv12_to_bgr(fake, 0, 4, 4, fake, None) == -1
    assert L.silent_nv12_to_bgr(fake, -2, 4, 4, fake, None) == -1
    assert L.silent_nv12_to_bgr(fake, 1, 0, 4, fake, None) == -1
    assert L.silent_nv12_to_bgr(fake, 1, 5, 4, fake, None) == -2
    assert L.silent_nv12_to_bgr(fake, 1, 4, 7, fake, None) == -2
    assert b"even" in L.silent_last_error()


def test_frame_format_and_shape_validation():
    from pysilent_b200 import LineEndPipeline, _ops
    from pysilent_b200.recognition_testing import LineEndDisplayer
    for bad in ("NV12", "yuv", "i420", None, 2):
        with pytest.raises(ValueError, match="frame_format"):
            LineEndPipeline(frame_format=bad)
        with pytest.raises(ValueError, match="frame_format"):
            LineEndDisplayer(frame_format=bad)
    assert LineEndPipeline().frame_format == "bgr"
    assert LineEndDisplayer(frame_format="nv12").frame_format == "nv12"
    pipe = LineEndPipeline(frame_format="nv12", output_size=(96, 64))
    disp = LineEndDisplayer(frame_format="nv12", output_size=(96, 64))
    good = random_nv12(1, 240, 320)
    for frames, what in ((good.astype(np.float32), "uint8"), (good[:-1], "even"), (good[:, :-1], "even"),
                         (good[0], "rank"), (good[None, None], "rank"), (good[:0], "rank")):
        with pytest.raises(ValueError, match=what):
            pipe.run_host(frames)
        with pytest.raises(ValueError, match=what):
            pipe.callback(frames)
        with pytest.raises(ValueError, match=what):
            pipe.run_frames(torch.from_numpy(np.ascontiguousarray(frames)))
        with pytest.raises(ValueError, match=what):
            _ops.nv12_to_bgr(torch.from_numpy(np.ascontiguousarray(frames)))
    with pytest.raises(ValueError, match="uint8"):
        pipe.run_host(good.astype(np.float16)[None])
    with pytest.raises(ValueError):
        disp.callback(good[None])                # a batch, not one frame
    with pytest.raises(ValueError, match="uint8"):
        disp.callback(good.astype(np.float32))
    with pytest.raises(ValueError):
        disp.run_clip(good)                      # a single frame, not a clip
    with pytest.raises(ValueError, match="even"):
        disp.run_clip(good[None, :-1])
    with pytest.raises(ValueError):
        disp.callback_clip(good)
    with pytest.raises(ValueError, match="uint8"):
        disp.callback_clip(good[None].astype(np.float32))


# ---- GPU ------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cuda(built_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert built_lib.silent_device_count() >= 1
    return torch


def _numpy(t):
    return t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def assert_bits(got, want, what):
    """Same dtype, shape and NaN mask; every other value has the same bit pattern."""
    g, w = _numpy(got), _numpy(want)
    assert g.dtype == w.dtype and g.shape == w.shape, (what, g.dtype, w.dtype, g.shape, w.shape)
    if g.dtype.kind != "f":
        assert np.array_equal(g, w), what
        return
    nan_g, nan_w = np.isnan(g), np.isnan(w)
    assert np.array_equal(nan_g, nan_w), "%s: NaN masks differ (%d vs %d)" % (what, nan_g.sum(), nan_w.sum())
    ints = np.uint16 if g.dtype == np.float16 else np.uint32
    same = g.view(ints) == w.view(ints)
    assert (same | nan_w).all(), "%s: %d of %d values differ" % (what, (~(same | nan_w)).sum(), same.size)


def assert_result(got, want, what):
    assert_bits(got.orient, want.orient, what + " orient")
    assert_bits(got.padded_line_end, want.padded_line_end, what + " padded_line_end")
    if want.gray is not None:
        assert_bits(got.gray, want.gray, what + " gray")
    if want.points is None:
        assert got.points is None
    else:
        assert np.array_equal(_numpy(got.points), _numpy(want.points)), what + " points"


def _pipes(**kw):
    from pysilent_b200 import LineEndPipeline
    return LineEndPipeline(frame_format="nv12", **kw), LineEndPipeline(**kw)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(2, 2), (480, 640), (1080, 1920), (768, 1366), (1920, 1080)])
def test_nv12_to_bgr_against_the_reference(h, w, cuda):
    from pysilent_b200 import _ops
    frames = np.stack([random_nv12(40 + h, h, w), structured_nv12(41, h, w) if h >= 10 else random_nv12(42, h, w)])
    want = nv12_to_bgr_reference(frames)
    got = _ops.nv12_to_bgr(_dev(frames))
    assert got.dtype == torch.uint8 and tuple(got.shape) == (2, h, w, 3) and got.is_contiguous()
    assert np.array_equal(got.cpu().numpy(), want), (h, w)
    assert np.array_equal(_ops.nv12_to_bgr(_dev(frames[1])).cpu().numpy(), want[1:])
    # a source that is not 16-byte aligned takes the byte-wise loads
    raw = torch.empty(frames.size + 1, dtype=torch.uint8, device="cuda")
    shifted = raw[1:].view(frames.shape)
    shifted.copy_(_dev(frames))
    assert np.array_equal(_ops.nv12_to_bgr(shifted).cpu().numpy(), want), (h, w, "unaligned")
    if h >= 10:
        black = want[1][(2 * h) // 5 + 2: (3 * h) // 5 - 2, (2 * w) // 5 + 2: (3 * w) // 5 - 2]
        assert black.size and not black.any()


@pytest.mark.gpu
def test_pyramid_build_on_an_nv12_plan(cuda):
    from pysilent_b200.util.zoom.from_image import PyramidPlan
    for (h, w), center, scale in (((480, 640), (96, 64), 1.5), ((768, 1366), (100, 66), 1.4)):
        frames = np.stack([random_nv12(50, h, w), structured_nv12(51, h, w), random_nv12(52, h, w)])
        nv12 = PyramidPlan((h, w, 3), torch.uint8, 3, center, scale, frame_format="nv12")
        bgr = PyramidPlan((h, w, 3), torch.uint8, 3, center, scale)
        assert nv12.levels == bgr.levels
        assert_bits(nv12.build(_dev(frames)), bgr.build(_dev(nv12_to_bgr_reference(frames))), "pyramid %s" % ((h, w),))


@pytest.mark.gpu
def test_run_frames_64_frames_1080p(cuda):
    p_nv, p_bgr = _pipes(zoom_ratio=SQRT2)
    frames = np.stack([structured_nv12(i, 1080, 1920) if i % 8 == 0 else random_nv12(100 + i, 1080, 1920)
                       for i in range(64)])
    got = p_nv.run_frames(_dev(frames))
    want = p_bgr.run_frames(_dev(nv12_to_bgr_reference(frames)))
    assert tuple(got.orient.shape) == tuple(want.orient.shape) and got.points.shape[0] > 0
    assert_result(got, want, "64 x 1080p")


@pytest.mark.gpu
def test_run_frames_odd_batch_single_frame_half_and_out_buffers(cuda):
    kw = dict(output_size=(96, 64), zoom_ratio=1.5)
    for out_dtype in (torch.float32, torch.float16):
        p_nv, p_bgr = _pipes(out_dtype=out_dtype, **kw)
        frames = np.stack([structured_nv12(60 + i, 480, 640) if i % 2 else random_nv12(60 + i, 480, 640)
                           for i in range(5)])
        bgr = _dev(nv12_to_bgr_reference(frames))
        assert_result(p_nv.run_frames(_dev(frames)), p_bgr.run_frames(bgr), "batch 5 %s" % out_dtype)
        assert_result(p_nv.run_frames(_dev(frames[1])), p_bgr.run_frames(bgr[1]), "single frame %s" % out_dtype)
        want = p_bgr.run_frames(bgr)
        orient = torch.empty(want.orient.shape, dtype=out_dtype, device="cuda")
        line_end = torch.empty_like(orient)
        points = torch.empty((4096, 4), dtype=torch.int64, device="cuda")
        count = torch.zeros(1, dtype=torch.int64, device="cuda")
        res = p_nv.run_frames(_dev(frames), out=(orient, line_end, points, count))
        assert res.orient is orient and res.padded_line_end is line_end
        assert_result(type(want)(orient, line_end, None, points[: int(count.item())]), want, "out= %s" % out_dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 6, 8, 12, 16])
def test_run_frames_banks(n, cuda):
    """Fused banks of 4, 8, 12 and 16 through the NV12 plan; width 6 through the conversion and the operator path."""
    for out_dtype in (torch.float32, torch.float16):
        p_nv, p_bgr = _pipes(output_size=(96, 64), zoom_ratio=1.5, orientations=n, out_dtype=out_dtype)
        frames = np.stack([structured_nv12(70 + i, 240, 320) if i % 2 else random_nv12(70 + i, 240, 320)
                           for i in range(3)])
        got = p_nv.run_frames(_dev(frames))
        assert got.orient.shape[-1] == n and got.orient.dtype == out_dtype
        assert_result(got, p_bgr.run_frames(_dev(nv12_to_bgr_reference(frames))), "bank %d %s" % (n, out_dtype))


def _tap_bounds(plan):
    rows, cols = [], []
    for s in range(plan.levels):
        iy, _, ix, _ = plan.level_tables(s)
        rows.append(iy[iy[:, 0] >= 0].min())
        cols.append(ix[ix[:, 0] >= 0].min())
    return min(rows), min(cols)


@pytest.mark.gpu
def test_crops_starting_on_odd_rows_and_columns(cuda):
    for (h, w), center, scale in (((482, 642), (72, 48), 1.3), ((486, 646), (100, 66), 1.7)):
        p_nv, p_bgr = _pipes(output_size=center, zoom_ratio=scale)
        frames = np.stack([structured_nv12(80, h, w), random_nv12(81, h, w)])
        y0, x0 = _tap_bounds(p_nv.plan_for(_dev(frames)))
        assert y0 % 2 == 1 or x0 % 2 == 1, (h, w, y0, x0)
        assert_result(p_nv.run_frames(_dev(frames)), p_bgr.run_frames(_dev(nv12_to_bgr_reference(frames))),
                      "odd crop %s" % ((h, w),))


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(768, 1366), (1920, 1080)])
def test_widths_off_16_take_the_frame_pair_path(h, w, cuda):
    """BGR rows of 3 * W bytes are not 16-byte aligned here, so BGR frames take the stand-alone pyramid_kernel; NV12
    frames are converted to padded rows and take the frame-pair kernel: one launch more than BGR's step (the
    conversion), and no pyramid_kernel."""
    L = _lib.lib()
    p_nv, p_bgr = _pipes(zoom_ratio=SQRT2)
    frames = np.stack([structured_nv12(90, h, w), random_nv12(91, h, w), random_nv12(92, h, w)])
    nv, bgr = _dev(frames), _dev(nv12_to_bgr_reference(frames))
    want, got = p_bgr.run_frames(bgr), p_nv.run_frames(nv)   # (plans built, workspaces reserved)
    assert_result(got, want, "%dx%d" % (h, w))
    torch.cuda.synchronize()
    c0 = L.silent_launch_count()
    p_bgr.run_frames(bgr)
    c1 = L.silent_launch_count()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        again = p_nv.run_frames(nv)
        torch.cuda.synchronize()
    c2 = L.silent_launch_count()
    assert c2 - c1 == (c1 - c0) + 1, (c1 - c0, c2 - c1)
    names = [e.name for e in prof.events()]
    assert any("nv12_to_bgr_kernel" in k for k in names) and any("pyramid_pair_kernel" in k for k in names), names
    assert not any("pyramid_kernel<" in k for k in names), names
    assert_result(again, want, "%dx%d again" % (h, w))


@pytest.mark.gpu
def test_run_host(cuda):
    frames = np.stack([structured_nv12(110, 300, 420), random_nv12(111, 300, 420), structured_nv12(112, 300, 420)])
    bgr = nv12_to_bgr_reference(frames)
    for out_dtype, out_np in ((torch.float32, np.float32), (torch.float16, np.float16)):
        p_nv, p_bgr = _pipes(output_size=(100, 66), zoom_ratio=1.4, out_dtype=out_dtype)
        want = p_bgr.run_host(bgr)
        got = p_nv.run_host(frames)
        assert got.orient.dtype == out_np
        assert_result(got, want, "run_host pageable %s" % out_dtype)
        pinned = torch.from_numpy(frames).pin_memory().numpy()
        assert_result(p_nv.run_host(pinned), want, "run_host pinned %s" % out_dtype)
        assert_result(p_nv.run_host(frames[1]), p_bgr.run_host(bgr[1]), "run_host one frame %s" % out_dtype)
        orient_out = np.full(want.orient.shape, 7, out_np)
        line_end_out = torch.empty(want.orient.shape, dtype=out_dtype).pin_memory().numpy()
        res = p_nv.run_host(frames, orient_out=orient_out, line_end_out=line_end_out)
        assert res.orient is orient_out and res.padded_line_end is line_end_out
        assert_result(res, want, "run_host caller arrays %s" % out_dtype)
        first = frames[0]
        cb_nv, cb_bgr = p_nv.callback(first), p_bgr.callback(bgr[0])
        assert cb_nv[0] is first and len(cb_nv[1]) == len(cb_bgr[1])
        for a, b in zip(cb_nv[1] + cb_nv[2], cb_bgr[1] + cb_bgr[2]):
            assert_bits(a, b, "callback level")
        assert np.array_equal(cb_nv[3], cb_bgr[3])
        small = np.ascontiguousarray(frames[:, :360, :320])   # (an NV12 array of a 240 x 320 image)
        for n in (8, 12, 6):
            b_nv, b_bgr = _pipes(output_size=(96, 64), zoom_ratio=1.5, orientations=n, out_dtype=out_dtype)
            assert_result(b_nv.run_host(small), b_bgr.run_host(nv12_to_bgr_reference(small)),
                          "run_host bank %d %s" % (n, out_dtype))


@pytest.mark.gpu
def test_displayer_callback_and_clips(cuda):
    """callback, run_clip (one and two cameras) and callback_clip against a BGR displayer fed the converted frames,
    interleaved on one state."""
    from pysilent_b200.recognition_testing import LineEndDisplayer
    kw = dict(output_size=(96, 64), zoom_ratio=1.5)
    d_nv, d_bgr = LineEndDisplayer(frame_format="nv12", **kw), LineEndDisplayer(**kw)
    h, w = 240, 320
    frames = np.stack([structured_nv12(120 + i, h, w) if i % 3 == 0 else random_nv12(120 + i, h, w) for i in range(7)])
    bgr = nv12_to_bgr_reference(frames)

    def same_callback(a, b, what):
        assert len(a) == len(b) == 7
        for x in range(1, 7):
            assert len(a[x]) == len(b[x])
            for y in range(len(a[x])):
                assert_bits(a[x][y], b[x][y], "%s tensor %d level %d" % (what, x, y))

    first = frames[0]
    out = d_nv.callback(first)
    assert out[0] is first
    same_callback(out, d_bgr.callback(bgr[0]), "callback 0")
    for a, b in zip(d_nv.run_clip(_dev(frames[1:4])), d_bgr.run_clip(_dev(bgr[1:4]))):
        assert_bits(a, b, "run_clip")
    same_callback(d_nv.callback(frames[4]), d_bgr.callback(bgr[4]), "callback 4")
    clip_nv, clip_bgr = d_nv.callback_clip(frames[5:7]), d_bgr.callback_clip(bgr[5:7])
    assert len(clip_nv) == len(clip_bgr) == 2
    for t in range(2):
        assert clip_nv[t][0] is frames[5 + t] or np.array_equal(clip_nv[t][0], frames[5 + t])
        same_callback(clip_nv[t], clip_bgr[t], "callback_clip %d" % t)
    assert torch.equal(d_nv.energy_values, d_bgr.energy_values)
    # two cameras: [T, S, H * 3 / 2, W]
    c_nv, c_bgr = LineEndDisplayer(frame_format="nv12", **kw), LineEndDisplayer(**kw)
    two = frames[:6].reshape((3, 2) + frames.shape[1:])
    for a, b in zip(c_nv.run_clip(_dev(two)), c_bgr.run_clip(_dev(nv12_to_bgr_reference(two)))):
        assert_bits(a, b, "run_clip two cameras")
    assert torch.equal(c_nv.energy_values, c_bgr.energy_values)
