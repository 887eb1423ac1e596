"""GPU parity: every CUDA entry point, called through the C ABI, against the oracle.

Bars (north_star): feature-point indices bit-exact; float32 responses within 1e-5 relative. Because center-surround
outputs are differences of large sums, "relative" is taken against the tensor's peak magnitude:
``|a - b| <= 1e-5 * max|ref|`` (SURVEY 7.3-4). Against the bit-defined C oracle (same canonical evaluation order) the
bar is stricter: bitwise equality of every finite value and identical NaN masks.
"""
import numpy as np
import pytest

from conftest import structured_frame, synthetic_frame

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

REL_TOL = 1e-5   # north_star tolerance


@pytest.fixture(scope="module", autouse=True)
def _need_cuda(built_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert built_lib.silent_device_count() >= 1


def assert_bits(actual, expected, what):
    a = actual.detach().cpu().numpy() if isinstance(actual, torch.Tensor) else np.asarray(actual)
    e = np.asarray(expected)
    assert a.shape == e.shape, (what, a.shape, e.shape)
    nan_a, nan_e = np.isnan(a), np.isnan(e)
    assert np.array_equal(nan_a, nan_e), "%s: NaN masks differ (%d vs %d)" % (what, nan_a.sum(), nan_e.sum())
    same = (a == e) | nan_e
    assert same.all(), "%s: %d of %d values differ from the bit-defined oracle, max |d| = %g" % (
        what, (~same).sum(), same.size, np.nanmax(np.abs(a - e)))


def assert_close(actual, expected, what, tol=REL_TOL, scale=None):
    """``scale``: magnitude of the OPERANDS when the result is a difference of much larger quantities (centroid
    distances are |centroid index - pixel index| with indices up to the level width)."""
    a = actual.detach().cpu().numpy() if isinstance(actual, torch.Tensor) else np.asarray(actual)
    e = np.asarray(expected)
    assert a.shape == e.shape, (what, a.shape, e.shape)
    assert np.array_equal(np.isnan(a), np.isnan(e)), "%s: NaN masks differ" % what
    peak = np.nanmax(np.abs(e)) if np.isfinite(e).any() else 1.0
    if scale is not None:
        peak = max(peak, scale)
    err = np.nanmax(np.abs(a - e)) if np.isfinite(e).any() else 0.0
    assert err <= tol * max(peak, 1e-30), "%s: max |d| = %g > %g * peak %g" % (what, err, tol, peak)


# ---- pyramid -----------------------------------------------------------------------------------------------------------

def test_pyramid_matches_reference_goldens(goldens, c_oracle):
    from pysilent_b200.util import zoom
    P = goldens["pyramid"]
    for name in [k[:-8] for k in P.files if k.endswith("_pyramid")]:
        img = P[name + "_image"]
        cw, ch, sc = P[name + "_params"]
        got = zoom.from_image(img, img.shape[2], [int(cw), int(ch)], float(sc))
        assert_close(got, P[name + "_pyramid"], "pyramid golden " + name)          # reference's own from_image output
        assert_bits(got, c_oracle.from_image(img, img.shape[2], [int(cw), int(ch)], float(sc)), "pyramid C " + name)
        got_f32 = zoom.from_image(img.astype(np.float32), img.shape[2], [int(cw), int(ch)], float(sc))
        assert_bits(got_f32, got.cpu().numpy(), "pyramid float32 frames " + name)


@pytest.mark.parametrize("shape,center,scale", [((480, 640), (288, 192), 1.3), ((480, 640), (288, 192), np.e ** .5),
                                                ((1080, 1920), (288, 192), 2 ** .5), ((720, 1280), (288, 192), 2 ** .5)])
def test_pyramid_full_size_bit_exact(shape, center, scale, c_oracle):
    from pysilent_b200.util import zoom
    frames = np.stack([synthetic_frame(2, i, *shape) for i in range(2)])
    got = zoom.from_image(frames, 3, center, scale)
    want = c_oracle.from_image(frames, 3, center, scale)
    assert_bits(got, want, "pyramid %s" % (shape,))


def test_pyramid_against_literal_oracle_and_properties():
    from oracle import silent_oracle as lit
    from pysilent_b200.util import zoom
    img = synthetic_frame(1, 0, 480, 640)
    got = zoom.from_image(img, 3, (288, 192), 1.3)
    assert tuple(got.shape) == (4, 192, 288, 3)
    assert_close(got, lit.from_image(img, 3, (288, 192), 1.3), "pyramid literal 640x480")
    # a constant image stays constant on every fully covered level (spline weights sum to 1)
    flat = np.full((480, 640, 3), 77, np.uint8)
    out = zoom.from_image(flat, 3, (288, 192), 1.3).cpu().numpy()
    assert np.abs(out - 77).max() < 1e-3
    # single channel and 4-channel frames taking 3 colours
    gray = zoom.from_image(img[:, :, :1], 1, (288, 192), 1.3)
    assert_bits(gray[..., 0], got[..., 0].cpu().numpy(), "1-channel pyramid")
    rgba = np.concatenate([img, img[:, :, :1]], axis=2)
    assert_bits(zoom.from_image(rgba, 3, (288, 192), 1.3), got.cpu().numpy(), "4-channel frame, 3 colours")


def test_pyramid_edge_cases():
    from pysilent_b200.util import zoom
    small = synthetic_frame(9, 0, 100, 150)
    out = zoom.from_image(small, 3, (288, 192), 1.5)      # image smaller than the centre: zero levels
    assert tuple(out.shape) == (0, 192, 288, 3)
    with pytest.raises(AssertionError):
        zoom.from_image(small, 3, (288, 192), 1.0)
    with pytest.raises(AssertionError):
        zoom.from_image(small, 0, (288, 192), 1.5)
    with pytest.raises(AssertionError):
        zoom.from_image(small, 3, (0, 192), 1.5)


# ---- per-operator kernels ------------------------------------------------------------------------------------------------

def _pyr(seed, n=3, h=40, w=56, c=3):
    return (np.random.RandomState(seed).rand(n, h, w, c) * 255).astype(np.float32)


def test_filter_callables_bit_exact(c_oracle, default_filters):
    from oracle import silent_oracle as lit
    from pysilent_b200 import filters
    x = _pyr(3)
    a = filters.rgc_filter(torch.from_numpy(x).cuda())
    assert_bits(a, c_oracle.conv2d(x, default_filters["rgc"], post=1), "rgc_filter")
    assert_close(a, lit.conv_relu(x, default_filters["rgc"]), "rgc_filter literal")
    b = filters.rgby_filter(a)
    b_ref = c_oracle.conv2d(a.cpu().numpy(), default_filters["rgby"], post=1)
    assert_bits(b, b_ref, "rgby_filter")
    assert_close(b, lit.conv_relu(a.cpu().numpy(), default_filters["rgby"]), "rgby_filter literal")
    d = filters.orientation_filter(b)
    c_ref = c_oracle.conv2d(b_ref, default_filters["stripe"], post=1)
    d_ref = c_oracle.regulate_tensor(c_ref, default_filters["blur"], 1.0, .1)
    assert_bits(d, d_ref, "orientation_filter")
    lit_c = lit.conv_relu(b_ref, default_filters["stripe"])
    assert_close(d, lit.regulate_tensor(lit_c, default_filters["blur"], 1.0, .1), "orientation_filter literal")
    d5 = filters.orientation_filter(b, blur_size=5)
    import pysilent_b200.constant_convolutions as cc
    assert_bits(d5, c_oracle.regulate_tensor(c_ref, cc.blur_tensor(2, lengths=5), 1.0, .1), "orientation_filter blur 5")
    # numpy input is accepted like the reference's get_dimensions allows
    assert_bits(filters.rgc_filter(x), a.cpu().numpy(), "rgc_filter(numpy)")


def test_apply_filter_generic_shapes(c_oracle, goldens):
    from pysilent_b200.util.apply_filter import apply_filter
    G = goldens["generators"]
    x3 = _pyr(4, n=2, h=33, w=47)
    for key in ("rgb_2d_end", "rgb_2d_edge", "rgb_2d_edge_time_diff", "rgb_2d_end_7x7", "rgby_2", "blur_2_default"):
        out = apply_filter(torch.from_numpy(x3).cuda(), G[key])
        assert_bits(out, c_oracle.conv2d(x3, G[key]), "apply_filter " + key)
    x8 = _pyr(5, n=2, h=21, w=30, c=8)
    for key in ("end_8", "stripe_8", "blur_8"):
        assert_bits(apply_filter(x8, G[key]), c_oracle.conv2d(x8, G[key]), "apply_filter " + key)
    # 3 -> 8 slice used by config C4, 1-pixel and 1-row tensors, NaN propagation through a dense conv
    w38 = G["stripe_8"][:, :, :3, :]
    assert_bits(apply_filter(x3, w38), c_oracle.conv2d(x3, w38), "apply_filter 3->8")
    tiny = _pyr(6, n=1, h=1, w=1)
    assert_bits(apply_filter(tiny, G["rgb_2d_end"]), c_oracle.conv2d(tiny, G["rgb_2d_end"]), "1x1 image")
    row = _pyr(7, n=2, h=1, w=70)
    assert_bits(apply_filter(row, G["rgb_2d_edge"]), c_oracle.conv2d(row, G["rgb_2d_edge"]), "1-row image")
    xn = x3.copy()
    xn[0, 5, 7, 1] = np.nan
    assert_bits(apply_filter(xn, G["rgb_2d_end"]), c_oracle.conv2d(xn, G["rgb_2d_end"]), "NaN input")


def test_regulate_pow_paths(c_oracle, default_filters):
    from pysilent_b200.util.regulator import regulate_tensor
    rs = np.random.RandomState(8)
    x = (rs.rand(2, 30, 41, 3) ** 6 * 0.2).astype(np.float32)     # blurred values straddle 1 -> both gain branches
    x[0, :12, :12] = 0                                             # exact zeros -> 0 * inf = NaN
    for root in (.1, .5, 1.0):
        got = regulate_tensor(x, default_filters["blur"], 1.0, root)
        want = c_oracle.regulate_tensor(x, default_filters["blur"], 1.0, root)
        assert np.isnan(want).any() and (want != x)[~np.isnan(want)].any()
        assert_bits(got, want, "regulate root %g" % root)
    from oracle import silent_oracle as lit
    assert_close(regulate_tensor(x, default_filters["blur"], 1.0, .1),
                 lit.regulate_tensor(x, default_filters["blur"], 1.0, .1), "regulate literal", tol=2e-5)


def test_pad_value_selection_ops(c_oracle):
    from oracle import silent_oracle as lit
    from pysilent_b200.util.selection import pad_inwards, max_value_indices_region, top_value_points
    from pysilent_b200.util.color import get_value_from_color
    x = _pyr(9, n=3, h=32, w=48)
    x[1, 10, 10, 0] = np.nan
    x[2] = 0                      # all-zero level: every pixel equals its region maximum
    pads = [[0, 0], [2, 2], [2, 2], [0, 0]]
    p = pad_inwards(x, pads)
    assert_bits(p, lit.pad_inwards(x, pads), "pad_inwards")
    assert_bits(pad_inwards(x, [[0, 0], [1, 3], [0, 5], [0, 0]]), lit.pad_inwards(x, [[0, 0], [1, 3], [0, 5], [0, 0]]),
                "pad_inwards asymmetric")
    g = get_value_from_color(p)
    g_ref = lit.get_value_from_color(lit.pad_inwards(x, pads))
    assert_bits(g, g_ref, "get_value_from_color")
    pts = max_value_indices_region(p, [1, 16, 24, 3], g).cpu().numpy()
    want = lit.max_value_indices_region(lit.pad_inwards(x, pads), [1, 16, 24, 3], g_ref)
    assert pts.dtype == np.int64 and np.array_equal(pts, want), (pts.shape, want.shape)
    assert (want[:, 0] == 2).sum() == 32 * 48 and (want[:, 0] == 1).sum() == 0    # zero level emits all, NaN level none
    c_pts, _ = c_oracle.max_value_indices_region(g_ref, (16, 24))
    assert np.array_equal(pts, c_pts)
    # value tensor computed internally, odd region split (3 x 3 overlapping windows)
    pts2 = max_value_indices_region(p, [1, 11, 16, 3]).cpu().numpy()
    assert np.array_equal(pts2, lit.max_value_indices_region(lit.pad_inwards(x, pads), [1, 11, 16, 3]))
    with pytest.raises(ValueError):
        max_value_indices_region(p, [1, 7.5, 24, 3], g)
    for pct in (.1, .5, 0.0):
        t = top_value_points(p, pct, g)
        assert_bits(t, lit.top_value_points(lit.pad_inwards(x, pads), pct, g_ref), "top_value_points %g" % pct)


# ---- fused stack ---------------------------------------------------------------------------------------------------------

def _check_stack(res, ref_c, ref_lit, what):
    assert_bits(res.orient, ref_c["orient"], what + " orient (C oracle)")
    assert_bits(res.padded_line_end, ref_c["padded"], what + " padded_line_end (C oracle)")
    if res.gray is not None:
        assert_bits(res.gray, ref_c["gray"], what + " gray (C oracle)")
    pts = res.points.cpu().numpy() if isinstance(res.points, torch.Tensor) else res.points
    assert np.array_equal(pts, ref_c["points"]), what + " points (C oracle)"
    if ref_lit is not None:
        assert_close(res.orient, ref_lit["orient"], what + " orient (literal)", tol=2e-5)
        assert_close(res.padded_line_end, ref_lit["padded"], what + " padded_line_end (literal)")
        assert np.array_equal(pts, ref_lit["points"]), what + " points (literal)"


def test_fused_stack_matches_reference_goldens(goldens, c_oracle, default_filters):
    from pysilent_b200 import LineEndPipeline
    S = goldens["stack"]
    for name in ("noise", "noise_odd", "natural", "flat"):
        pyr = S[name + "_pyramid"]
        pipe = LineEndPipeline(output_size=(pyr.shape[2], pyr.shape[1]))
        res = pipe.run(pyr)
        ref_c = c_oracle.line_end_stack(pyr, default_filters)
        ref_lit = {k: S[name + "_" + k] for k in ("orient", "padded", "points")}     # reference code on the TF-1 shim
        _check_stack(res, ref_c, ref_lit, "golden " + name)
        unfused = pipe.run_unfused(pyr)   # operator by operator: one (ky, ci, kx) chain per output
        _check_stack(unfused, c_oracle.line_end_stack(pyr, default_filters, order="operator"), None,
                     "golden unfused " + name)


@pytest.mark.parametrize("seed,n,h,w", [(31, 2, 64, 96), (32, 1, 37, 53), (33, 3, 192, 288), (34, 2, 5, 9)])
def test_fused_stack_bit_exact_random(seed, n, h, w, c_oracle, default_filters):
    from oracle import silent_oracle as lit
    from pysilent_b200 import LineEndPipeline
    pyr = _pyr(seed, n, h, w)
    pipe = LineEndPipeline(output_size=(w - w % 2, h - h % 2))
    orient, line_end, gray = __import__("pysilent_b200")._ops.stack_fused(pyr, pipe.stack_weights())
    ref = c_oracle.line_end_stack(pyr, default_filters)
    assert_bits(orient, ref["orient"], "orient")
    assert_bits(line_end, ref["padded"], "padded_line_end")
    assert_bits(gray, ref["gray"], "gray")
    ref_lit = lit.line_end_stack(pyr, default_filters)
    assert_close(orient, ref_lit["orient"], "orient literal")
    assert_close(line_end, ref_lit["padded"], "padded literal")


@pytest.mark.parametrize("seed,n,h,w", [(35, 2, 64, 96), (36, 3, 37, 53), (37, 2, 30, 100)])
def test_fused_stack_dense_variants_bit_exact(seed, n, h, w, c_oracle, default_filters):
    """Weights without the generators' structure run the dense variants of both kernels (stack_a without its depthwise
    rgc + shared-surround rgby form, stack_b without its symmetric-stripe + own / other end form): bitwise against the
    oracle, which takes the same dispatch. The second weight set keeps the depthwise rgc, rgby_3's zero pattern and
    stack_b's structure and breaks only the shared surround: stack_a runs dense there, like the oracle. The widths cover
    the three routes a staged tile leaves by: tile stores, bulk rows, element-wise."""
    from pysilent_b200 import _lib, _ops
    L = c_oracle.lib()
    f32 = lambda a: np.ascontiguousarray(a, np.float32)
    dense = {k: np.array(v, copy=True) for k, v in default_filters.items()}
    dense["rgc"][1, 1, 0, 1] = 0.05          # not depthwise
    dense["rgby"][0, 0, 1, 2] *= 1.5         # not the shared surround (as in test_c_oracle_fused_order_uses_the_structures) ...
    dense["rgby"][0, 0, 1, 1] = 0.05         # ... nor the zero pattern
    dense["end"][2, 1, 0, 1] += 0.01         # not own / other
    assert not L.so_depthwise3(f32(dense["rgc"])) and not L.so_rgby_shared(f32(dense["rgby"]))
    assert not L.so_end_ownoth(f32(dense["end"]))
    zeros = {k: np.array(v, copy=True) for k, v in default_filters.items()}
    zeros["rgby"][0, 0, 1, 2] *= 1.5         # not the shared surround; every structural zero of rgby_3 stays zero
    assert np.array_equal(zeros["rgby"] == 0, default_filters["rgby"] == 0)
    assert L.so_depthwise3(f32(zeros["rgc"])) and not L.so_rgby_shared(f32(zeros["rgby"]))
    assert L.so_stripe_sym180(f32(zeros["stripe"])) and L.so_end_ownoth(f32(zeros["end"]))
    pyr = _pyr(seed, n, h, w)
    for name, f in (("dense", dense), ("rgby_3 zero pattern", zeros)):
        orient, line_end, gray = _ops.stack_fused(pyr, _lib.make_stack_weights(f["rgc"], f["rgby"], f["stripe"],
                                                                               f["blur"], f["end"]))
        ref = c_oracle.line_end_stack(pyr, f)
        assert_bits(orient, ref["orient"], "orient, " + name)
        assert_bits(line_end, ref["padded"], "padded_line_end, " + name)
        assert_bits(gray, ref["gray"], "gray, " + name)


def test_fused_stack_rejects_unstructured_weights():
    from pysilent_b200 import LineEndPipeline, _lib, _ops
    pipe = LineEndPipeline()
    f = pipe.filters()
    f["stripe"] = f["stripe"].copy()
    f["stripe"][0, 0, 1, 0] += 1.0
    w = _lib.make_stack_weights(f["rgc"], f["rgby"], f["stripe"], f["blur"], f["end"])
    with pytest.raises(RuntimeError, match="stripe filter differs"):
        _ops.stack_fused(_pyr(1, 1, 16, 16), w)


# ---- whole pipeline ------------------------------------------------------------------------------------------------------

def _oracle_pipeline(c_oracle, frames, center, scale, filters):
    pyr = c_oracle.from_image(frames, 3, center, scale)
    return pyr, c_oracle.line_end_stack(pyr, filters)


@pytest.mark.parametrize("config,shape,scale,batch", [(1, (480, 640), 1.3, 1), (2, (1080, 1920), 2 ** .5, 1),
                                                      (5, (720, 1280), 2 ** .5, 3)])
def test_pipeline_baseline_configs_bit_exact(config, shape, scale, batch, c_oracle, default_filters):
    """BASELINE configs C1 / C2 / C5 (frame shapes and level counts), device-resident and host-buffer entry points."""
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([synthetic_frame(config, i, *shape) for i in range(batch)])
    pipe = LineEndPipeline(zoom_ratio=scale)
    pyr, ref = _oracle_pipeline(c_oracle, frames, (288, 192), scale, default_filters)
    res = pipe.run_frames(torch.from_numpy(frames).cuda())
    assert tuple(res.orient.shape) == pyr.shape
    _check_stack(res, ref, None, "config %d device" % config)
    host = pipe.run_host(frames)
    _check_stack(host, ref, None, "config %d host" % config)
    cb = pipe.callback(frames[0])
    assert cb[0] is frames[0] or np.array_equal(cb[0], frames[0])
    assert len(cb[1]) == pyr.shape[0] // batch and np.array_equal(cb[1][0], ref["orient"][0], equal_nan=True)


@pytest.mark.parametrize("shape,scale", [((2000, 112), 1.5), ((240, 1920), 2 ** .5), ((96, 1600), 1.7)])
def test_pipeline_extreme_aspect_frames_bit_exact(shape, scale, c_oracle, default_filters):
    """Frames far from the level aspect ratio: the coarse crops leave the frame on one axis, so whole x tiles of the
    pyramid kernel have no defined column (tile without a word span) and hundreds of output rows are undefined (zero
    rows). Device and host entry points bitwise against the oracle, odd batch."""
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([synthetic_frame(7, i, *shape) for i in range(3)])
    pipe = LineEndPipeline(zoom_ratio=scale)
    pyr, ref = _oracle_pipeline(c_oracle, frames, (288, 192), scale, default_filters)
    assert (pyr == 0).all(axis=(2, 3)).any() or (pyr == 0).all(axis=(1, 3)).any()   # undefined rows or columns exist
    res = pipe.run_frames(torch.from_numpy(frames).cuda())
    _check_stack(res, ref, None, "extreme aspect %s device" % (shape,))
    _check_stack(pipe.run_host(frames), ref, None, "extreme aspect %s host" % (shape,))


def test_pipeline_structured_frames_nan_and_gain_paths(c_oracle, default_filters):
    from oracle import silent_oracle as lit
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([structured_frame(41 + i, 480, 640) for i in range(2)])
    pipe = LineEndPipeline(zoom_ratio=1.3)
    pyr, ref = _oracle_pipeline(c_oracle, frames, (288, 192), 1.3, default_filters)
    assert np.isnan(ref["orient"]).any(), "the structured frame must exercise the 0 * inf path"
    res = pipe.run_frames(torch.from_numpy(frames).cuda())
    ref_lit = lit.line_end_stack(lit.from_image(frames[0], 3, (288, 192), 1.3), default_filters)
    _check_stack(res, ref, None, "structured")
    n0 = ref_lit["orient"].shape[0]
    assert_close(res.orient[:n0], ref_lit["orient"], "structured orient literal", tol=2e-5)
    lit_pts = ref_lit["points"]
    got_pts = res.points.cpu().numpy()
    assert np.array_equal(got_pts[got_pts[:, 0] < n0], lit_pts)


def test_pipeline_properties_at_full_size(default_filters):
    """Size-independent properties on the BASELINE C3 shape (1080p, batch 8): batch independence, determinism,
    idempotence of the mask, point rows sorted and inside the border."""
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([synthetic_frame(3, i, 1080, 1920) for i in range(8)])
    pipe = LineEndPipeline(zoom_ratio=2 ** .5)
    dev = torch.from_numpy(frames).cuda()
    full = pipe.run_frames(dev)
    again = pipe.run_frames(dev)
    assert torch.equal(full.orient, again.orient) and torch.equal(full.points, again.points)
    L = full.orient.shape[0] // 8
    for i in (0, 5):
        one = pipe.run_frames(dev[i:i + 1])
        assert torch.equal(one.orient, full.orient[i * L:(i + 1) * L])
        assert torch.equal(one.padded_line_end, full.padded_line_end[i * L:(i + 1) * L])
        sel = full.points[(full.points[:, 0] >= i * L) & (full.points[:, 0] < (i + 1) * L)].clone()
        sel[:, 0] -= i * L
        assert torch.equal(one.points, sel)
    pts = full.points.cpu().numpy()
    key = (pts[:, 0] * 192 + pts[:, 1]) * 288 + pts[:, 2]
    assert (np.diff(key) > 0).all() and (pts[:, 3] == 0).all()
    p = full.padded_line_end
    assert float(p[:, :2].abs().max()) == 0 and float(p[:, :, -2:].abs().max()) == 0
    assert float(p.max()) <= 255.0 and float(p.min()) >= 0.0 and float(full.orient.min()) >= 0.0
    from pysilent_b200.util.selection import pad_inwards
    assert torch.equal(pad_inwards(p, [[0, 0], [2, 2], [2, 2], [0, 0]]), p)


@pytest.mark.parametrize("batch", [64, 63])
def test_pipeline_config3_full_batch_against_oracle(batch, c_oracle, default_filters):
    """The headline config itself (C3: 1080p, 6 levels, batch 64) against the bit-defined oracle: first, middle and last
    frames (values, NaN masks, gray-derived points), device-resident and host-buffer entry points; batch 63 leaves a lone
    frame in the last frame pair."""
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([synthetic_frame(3, i, 1080, 1920) for i in range(batch)])
    pipe = LineEndPipeline(zoom_ratio=2 ** .5)
    res = pipe.run_frames(torch.from_numpy(frames).cuda())
    host = pipe.run_host(frames) if batch == 64 else None
    L = 6
    assert tuple(res.orient.shape) == (batch * L, 192, 288, 3)
    pts = res.points.cpu().numpy()
    for i in (0, 31, batch - 2, batch - 1):
        pyr, ref = _oracle_pipeline(c_oracle, frames[i:i + 1], (288, 192), 2 ** .5, default_filters)
        assert pyr.shape[0] == L
        sl = slice(i * L, (i + 1) * L)
        assert_bits(res.orient[sl], ref["orient"], "C3 frame %d orient" % i)
        assert_bits(res.padded_line_end[sl], ref["padded"], "C3 frame %d padded_line_end" % i)
        sel = pts[(pts[:, 0] >= i * L) & (pts[:, 0] < (i + 1) * L)].copy()
        sel[:, 0] -= i * L
        assert np.array_equal(sel, ref["points"]), "C3 frame %d points" % i
        if host is not None:
            assert_bits(host.orient[sl], ref["orient"], "C3 host frame %d orient" % i)
            assert_bits(host.padded_line_end[sl], ref["padded"], "C3 host frame %d padded_line_end" % i)
    if host is not None:
        assert np.array_equal(host.points, pts)


def test_run_host_returns_every_point():
    """run_host never truncates the feature points: a too-small capacity is retried with the reported count, and a
    capacity beyond the plan's own point buffer grows it."""
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([synthetic_frame(1, i, 240, 320) for i in range(2)])
    pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=1.5)
    dev = pipe.run_frames(torch.from_numpy(frames).cuda()).points.cpu().numpy()
    assert len(dev) > 1
    assert np.array_equal(pipe.run_host(frames, points_capacity=1).points, dev)
    assert np.array_equal(pipe.run_host(frames, points_capacity=200000).points, dev)


def test_two_devices_in_one_process(default_filters):
    """One process, two GPUs (camera threads on different devices): per-device kernel attributes (the pyramid kernel's
    dynamic shared memory at 1080p exceeds the 48 KB default) must be set on each device."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([synthetic_frame(2, i, 1080, 1920) for i in range(2)])
    outs = []
    for d in (0, 1):
        pipe = LineEndPipeline(zoom_ratio=2 ** .5, device="cuda:%d" % d)
        with torch.cuda.device(d):
            res = pipe.run_frames(torch.from_numpy(frames).to("cuda:%d" % d))
            outs.append((res.orient.cpu(), res.padded_line_end.cpu(), res.points.cpu()))
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)


def test_fused_stack_routes_non_finite_input(c_oracle, default_filters):
    """``run(pyramid)`` on input with NaN / Inf: the fused kernels assume finite input (they skip exact-zero weights and
    shortcut the regulator), so the pipeline takes the per-operator path, which propagates like the reference graph."""
    from pysilent_b200 import LineEndPipeline
    pyr = _pyr(77, 2, 40, 56)
    pyr[0, 10, 12, 1] = np.nan
    pyr[1, 20, 30, 0] = np.inf
    pipe = LineEndPipeline(output_size=(56, 40))
    res = pipe.run(pyr)
    ref = c_oracle.line_end_stack(pyr, default_filters, order="operator")
    assert np.isnan(ref["orient"]).any()
    _check_stack(res, ref, None, "non-finite pyramid")
    clean = _pyr(77, 2, 40, 56)
    _check_stack(pipe.run(clean), c_oracle.line_end_stack(clean, default_filters), None, "finite pyramid (fused)")


# ---- BASELINE config C4: 8-orientation bank, 8-level 4K pyramid ----------------------------------------------------------

def _oracle_bank(c_oracle, pyr, f, region, order="fused"):
    """uint8 frames take the fused bank path (rgc / rgby in the fused order); ``run_bank`` on a pyramid goes operator by
    operator."""
    return c_oracle.bank_stack(pyr, f, region, order=order)


def test_orientation_bank_config4_bit_exact(c_oracle, goldens):
    """C4's filter bank (8 orientations: stripe 3->8, blur 8->8, end 8->8) on a small frame: every stage bit-equal to the
    C oracle composed operator by operator, bank weights equal to the reference generators' own output."""
    from oracle import silent_oracle as lit
    from pysilent_b200 import LineEndPipeline
    pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=2 ** .5, orientations=8)
    f = pipe.bank_filters()
    G = goldens["generators"]
    assert np.array_equal(f["stripe"], G["stripe_8"][:, :, :3, :]) and np.array_equal(f["end"], G["end_8"])
    assert np.array_equal(f["blur"], G["blur_8"])
    frames = np.stack([structured_frame(70 + i, 300, 432) for i in range(3)])   # odd batch: a lone frame in the last pair
    pyr = c_oracle.from_image(frames, 3, (96, 64), 2 ** .5)
    ref = _oracle_bank(c_oracle, pyr, f, (32, 48))
    res = pipe.run_frames(torch.from_numpy(frames).cuda())
    assert tuple(res.orient.shape) == pyr.shape[:3] + (8,)
    _check_stack(res, ref, None, "config 4 bank")
    per_op = pipe.run_bank(pyr)   # the same bank operator by operator (any channel count / structure)
    _check_stack(per_op, _oracle_bank(c_oracle, pyr, f, (32, 48), order="operator"), None, "config 4 bank, per operator")
    lit_orient = lit.regulate_tensor(lit.conv_relu(lit.conv_relu(lit.conv_relu(pyr, f["rgc"]), f["rgby"]), f["stripe"]),
                                     f["blur"], 1.0, .1)
    assert_close(res.orient, lit_orient, "config 4 orient literal", tol=2e-5)


def test_orientation_bank_config4_full_size_properties():
    """C4 at its named shape (3840x2160, scale sqrt2 -> 8 levels, 8 orientations): level count, batch independence,
    determinism, value ranges, sorted point rows."""
    from pysilent_b200 import LineEndPipeline
    frames = np.stack([synthetic_frame(4, i, 2160, 3840) for i in range(2)])
    pipe = LineEndPipeline(zoom_ratio=2 ** .5, orientations=8)
    dev = torch.from_numpy(frames).cuda()
    full = pipe.run_frames(dev)
    assert tuple(full.orient.shape) == (16, 192, 288, 8) and tuple(full.padded_line_end.shape) == (16, 192, 288, 8)
    one = pipe.run_frames(dev[1:2])
    assert torch.equal(one.orient, full.orient[8:]) and torch.equal(one.padded_line_end, full.padded_line_end[8:])
    again = pipe.run_frames(dev)
    assert torch.equal(again.padded_line_end, full.padded_line_end) and torch.equal(again.points, full.points)
    p = full.padded_line_end
    assert float(p[:, :2].abs().max()) == 0 and float(p[:, :, -2:].abs().max()) == 0
    assert float(p.max()) <= 255.0 and float(p.min()) >= 0.0 and float(full.orient.min()) >= 0.0
    pts = full.points.cpu().numpy()
    key = (pts[:, 0] * 192 + pts[:, 1]) * 288 + pts[:, 2]
    assert len(pts) > 0 and (np.diff(key) > 0).all()


def test_orientation_bank_config4_4k_against_oracle(c_oracle):
    """C4 at its named frame shape: one 3840x2160 frame, all 8 levels, 8 orientations, against the bit-defined oracle."""
    from pysilent_b200 import LineEndPipeline
    frame = synthetic_frame(4, 0, 2160, 3840)
    pipe = LineEndPipeline(zoom_ratio=2 ** .5, orientations=8)
    res = pipe.run_frames(torch.from_numpy(frame[None]).cuda())
    pyr = c_oracle.from_image(frame[None], 3, (288, 192), 2 ** .5)
    assert pyr.shape == (8, 192, 288, 3)
    ref = _oracle_bank(c_oracle, pyr, pipe.bank_filters(), (96, 144))
    _check_stack(res, ref, None, "config 4 at 4K")


# ---- BASELINE config C5: many 720p streams; host-buffer entry point from several camera threads --------------------------

def test_multi_stream_config5_chunked_host_path(c_oracle, default_filters):
    """C5 shape (1280x720, 5 levels): a batch of streams through the chunked, overlapped host-buffer call equals the
    device-resident call and the oracle, for batches that do and do not fill whole chunks (odd batch: a lone frame in
    the last pair)."""
    from pysilent_b200 import LineEndPipeline
    pipe = LineEndPipeline(zoom_ratio=2 ** .5)
    frames = np.stack([synthetic_frame(5, i, 720, 1280) for i in range(37)])
    dev = pipe.run_frames(torch.from_numpy(frames).cuda())
    host = pipe.run_host(frames)
    assert np.array_equal(host.orient, dev.orient.cpu().numpy(), equal_nan=True)
    assert np.array_equal(host.padded_line_end, dev.padded_line_end.cpu().numpy(), equal_nan=True)
    assert np.array_equal(host.points, dev.points.cpu().numpy())
    pyr, ref = _oracle_pipeline(c_oracle, frames[35:37], (288, 192), 2 ** .5, default_filters)
    L = pyr.shape[0] // 2
    assert np.array_equal(host.orient[35 * L:], ref["orient"], equal_nan=True)
    sel = host.points[host.points[:, 0] >= 35 * L].copy()
    sel[:, 0] -= 35 * L
    assert np.array_equal(sel, ref["points"])
    pinned = torch.from_numpy(frames[:6]).pin_memory()
    o = torch.empty((6 * L, 192, 288, 3), dtype=torch.float32).pin_memory()
    l = torch.empty_like(o).pin_memory()
    part = pipe.run_host(pinned.numpy(), o.numpy(), l.numpy())
    assert np.array_equal(part.orient, host.orient[:6 * L], equal_nan=True)
    assert np.array_equal(part.padded_line_end, host.padded_line_end[:6 * L], equal_nan=True)


def test_callback_from_camera_threads(c_oracle, default_filters):
    """The reference calls ``callback`` on one thread per camera (SURVEY 8(b)): concurrent calls from non-main threads,
    one pipeline per camera, give the single-threaded results."""
    import threading
    from pysilent_b200 import LineEndPipeline
    frames = [synthetic_frame(1, i, 480, 640) for i in range(4)]
    want = []
    for fr in frames:
        _, ref = _oracle_pipeline(c_oracle, fr[None], (288, 192), 1.3, default_filters)
        want.append(ref)
    got = [None] * 4
    errors = []

    def camera(i):
        try:
            torch.cuda.set_device(0)
            pipe = LineEndPipeline(zoom_ratio=1.3)
            with torch.cuda.stream(torch.cuda.Stream()):
                for _ in range(3):
                    got[i] = pipe.callback(frames[i], cam_id=i)
        except Exception as exc:   # surfaced below: an exception in a thread would otherwise pass silently
            errors.append(exc)

    threads = [threading.Thread(target=camera, args=(i,)) for i in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i in range(4):
        assert np.array_equal(np.stack(got[i][1]), want[i]["orient"], equal_nan=True)
        assert np.array_equal(np.stack(got[i][2]), want[i]["padded"], equal_nan=True)
        assert np.array_equal(got[i][3], want[i]["points"])


# ---- SURVEY 8(f) next rows: centroids, boosting, the reference driver's six display tensors -------------------------------

def test_centroids_resize_boosting_operators_bit_exact(c_oracle):
    from oracle import silent_oracle as lit
    from pysilent_b200.util import get_centroids
    from pysilent_b200.util.centroids import get_centroids_array
    from pysilent_b200.util.energy import get_boosting, initialize_boosting
    from pysilent_b200 import _ops
    rs = np.random.RandomState(51)
    for n, h, w, region in ((2, 12, 18, [1, 3, 3]), (3, 13, 17, [1, 3, 3]), (1, 116, 174, [1, 3, 3]), (2, 20, 31, [1, 2, 4])):
        v = rs.rand(n, h, w, 1).astype(np.float32)
        v[0, :5, :7] = 0                                # empty blocks: 0 / 0 = NaN centroids
        cent, total = get_centroids(v, region)
        want_c, want_t, want_arr = c_oracle.get_centroids(v, region)
        assert_bits(cent, want_c, "get_centroids %s" % ((n, h, w),))
        assert_bits(total, want_t, "total_pool")
        assert_bits(get_centroids_array(v, region), want_arr, "get_centroids_array")
        lit_c, lit_t = lit.get_centroids(v, region)
        assert np.isnan(lit_c).any()
        assert_close(cent, lit_c, "get_centroids literal", scale=max(h, w))
        assert_close(total, lit_t, "total_pool literal")
        assert_bits(_ops.resize_nearest(v, 7, 11), c_oracle.resize_nearest(v, (7, 11)), "resize_nearest")
        assert_bits(_ops.resize_nearest(v, 7, 11), lit.resize_nearest_neighbor(v, (7, 11)), "resize_nearest literal")
    with pytest.raises(ValueError):
        get_centroids(v, [1, 2.5, 3])
    # boosting: five frames of a still camera, then a changed input; all three recovery selections
    imp = (rs.rand(2, 16, 24, 1) * 60).astype(np.float32)
    imp[1, 4:9, 4:9] = 0
    for kw, mode in ((dict(), 1), (dict(input_based_recovery=True, constant_recovery=False), 2),
                     (dict(input_based_recovery=True), 3)):
        energy = initialize_boosting(imp)
        e_ref = np.full_like(imp, 8)
        e_lit = e_ref.copy()
        for step in range(6):
            x = imp if step < 4 else imp[:, ::-1].copy()
            fired, state = get_boosting(x, energy, **kw)
            f_ref, e_ref = c_oracle.get_boosting(x, e_ref, recovery_mode=mode)
            assert state is energy
            assert_bits(fired, f_ref, "has_fired step %d mode %d" % (step, mode))
            assert_bits(energy, e_ref, "energy step %d mode %d" % (step, mode))
            f_lit, e_lit = lit.get_boosting(x, e_lit, **kw)
            assert_bits(fired, f_lit, "has_fired literal")
            assert_close(energy, e_lit, "energy literal")
    with pytest.raises(ValueError):
        get_boosting(imp, energy, input_based_recovery=False, constant_recovery=False)


def test_displayer_matches_reference_goldens(goldens, c_oracle):
    """The six fetched tensors of three consecutive frames on the reference's golden pyramids.

    (a) ``LineEndDisplayer.run`` (pyramid -> everything) bitwise against the C oracle. (b) The display operators fed the
    GOLDEN gray / padded tensors against the reference's own centroid / boosting code executed on the TF-1 shim
    (tests/golden/display.npz), to the north-star tolerance with identical fired cells. (b) isolates the display
    operators: a block centroid sum(idx * v) / sum(v) is ill-conditioned where a block is almost empty, so float32
    rounding noise of the upstream filter stack (1e-5 of its peak) may move such centroids arbitrarily."""
    from pysilent_b200 import LineEndDisplayer
    S = goldens["stack"]
    D = np.load(__import__("os").path.join(__import__("conftest").GOLDEN, "display.npz"))
    for name in ("noise", "natural", "flat"):
        pyr = S[name + "_pyramid"]
        disp = LineEndDisplayer(output_size=(pyr.shape[2], pyr.shape[1]))
        iso = LineEndDisplayer(output_size=(pyr.shape[2], pyr.shape[1]))
        ref = c_oracle.line_end_stack(pyr, disp.filters())
        energy = np.full((pyr.shape[0], -(-pyr.shape[1] // 3), -(-pyr.shape[2] // 3), 1), 8, np.float32)
        g_orient, g_padded, g_gray = (torch.from_numpy(S[name + k]).cuda() for k in ("_orient", "_padded", "_gray"))
        for step in range(3):
            got = disp.run(pyr)
            want, energy = c_oracle.display_tensors(ref["orient"], ref["padded"], ref["gray"], energy)
            assert len(got) == 6
            for i, (g, wv) in enumerate(zip(got, want)):
                assert_bits(g, wv, "%s step %d tensor %d" % (name, step, i))
            got_iso = iso.display_tensors(g_orient, g_padded, g_gray)
            for key, i in (("centroids", 1), ("centroids2", 2), ("fired", 3), ("update", 4)):
                gold = D["%s_step%d_%s" % (name, step, key)]
                assert_close(got_iso[i], gold, "%s step %d %s vs reference code" % (name, step, key),
                             scale=255.0 * max(pyr.shape[1:3]) if key.startswith("centroids") else None)
            assert np.array_equal(got_iso[3].cpu().numpy() > 0, D["%s_step%d_fired" % (name, step)] > 0)
            assert_close(iso.energy_values, D["%s_step%d_energy" % (name, step)], "energy vs reference code")


@pytest.mark.parametrize("h,w,region", [(192, 288, 3), (100, 149, 3), (37, 53, 4), (64, 96, 2)])
def test_display_tensors_fused_matches_operator_chain(h, w, region):
    """``silent_display_tensors`` (two launches) against the chain of stand-alone operators the reference graph is written
    as (recognition_testing.py:79-100), bitwise, over three frames of boosting state -- on level shapes the region does not
    divide (ragged last blocks, pixel -> block through the float nearest-neighbour scale) and with empty blocks (0 / 0)."""
    from pysilent_b200 import LineEndDisplayer
    rs = np.random.RandomState(h * 7 + w)
    n = 3
    a, b = LineEndDisplayer(), LineEndDisplayer()
    a.centroid_region_shape = b.centroid_region_shape = [1, region, region]
    for step in range(3):
        gray = rs.uniform(0, 255, size=(n, h, w, 1)).astype(np.float32)
        gray[rs.uniform(size=gray.shape) < 0.4] = 0.0
        gray[0, : 3 * region, : 5 * region] = 0.0               # empty blocks: centroid 0 / 0 = NaN, importance 0
        gray[1] = 0.0 if step == 1 else gray[1]
        g = torch.from_numpy(gray).cuda()
        orient = torch.zeros((n, h, w, 3), device="cuda")
        padded = torch.zeros((n, h, w, 3), device="cuda")
        fused = a.display_tensors(orient, padded, g, fused=True)
        chain = b.display_tensors(orient, padded, g, fused=False)
        for i in (1, 2, 3, 4):
            assert tuple(fused[i].shape) == tuple(chain[i].shape), (i, fused[i].shape, chain[i].shape)
            assert_bits(fused[i], chain[i].cpu().numpy(), "step %d display tensor %d" % (step, i))
        assert_bits(a.energy_values, b.energy_values.cpu().numpy(), "boosting state after step %d" % step)
    assert np.isnan(fused[1].cpu().numpy()).any()


def test_displayer_callback_structure_and_state(c_oracle, default_filters):
    """callback(frame, cam_id) returns ``[frame] + 6 lists of per-level images`` (recognition_testing.py:144); the
    boosting state persists across frames and is reset when the frame shape changes; display() scales by 1/255."""
    from pysilent_b200 import LineEndDisplayer
    disp = LineEndDisplayer(zoom_ratio=1.3)
    frame = synthetic_frame(1, 0, 480, 640)
    pyr, ref = _oracle_pipeline(c_oracle, frame[None], (288, 192), 1.3, default_filters)
    L = pyr.shape[0]
    energy = np.full((L, 64, 96, 1), 8, np.float32)
    for step in range(2):
        out = disp.callback(frame, cam_id=0)
        want, energy = c_oracle.display_tensors(ref["orient"], ref["padded"], ref["gray"], energy)
        assert out[0] is frame and len(out) == 7 and all(len(out[1 + x]) == L for x in range(6))
        for x in range(6):
            assert_bits(np.stack(out[1 + x]), want[x], "callback step %d tensor %d" % (step, x))
    assert out[1][0].shape == (192, 288, 3) and out[2][0].shape == (192, 288, 1) and out[3][0].shape == (116, 174, 1)
    assert out[4][0].shape == (64, 96, 3) and out[5][0].shape == (64, 96, 3)
    small = synthetic_frame(1, 1, 360, 480)
    disp.callback(small)
    assert tuple(disp.energy_values.shape)[0] != L or float(disp.energy_values.max()) <= 1.0
    _, ref_s = _oracle_pipeline(c_oracle, small[None], (288, 192), 1.3, default_filters)
    e0 = np.full((ref_s["gray"].shape[0], 64, 96, 1), 8, np.float32)
    want_s, e1 = c_oracle.display_tensors(ref_s["orient"], ref_s["padded"], ref_s["gray"], e0)
    assert_bits(disp.energy_values, e1, "state re-initialised on shape change")
    shown = disp.display(small)
    assert len(shown) == 7 and float(np.nanmax(shown[6])) <= 1.0


# ---- multi-GPU exchange: the feature-point gather -------------------------------------------------------------------------

def test_point_gather_pack_and_single_rank_path():
    """silent_pack_points + PointGather on one GPU (world 1): level ids rebased to global frame order, rows beyond the
    count zeroed, count row last; repeated submits reuse the two slots."""
    from pysilent_b200.distributed import PointGather
    rs = np.random.RandomState(77)
    cap, levels = 48, 6
    g = PointGather(cap, levels, torch.device("cuda", 0))
    for step, k_valid in enumerate((5, 0, 48, 60, 17)):
        pts = torch.from_numpy(rs.randint(0, 190, size=(64, 4)).astype(np.int64)).cuda()
        count = torch.tensor([k_valid], dtype=torch.int64, device="cuda")
        slot = g.submit(pts, count, frame_offset=3 + step)
        got, counts = g.result(slot)
        keep = min(k_valid, cap)
        want = pts[:keep].clone()
        want[:, 0] += (3 + step) * levels
        assert int(counts[0]) == k_valid and torch.equal(got, want)
        send = g.send[slot].cpu().numpy()
        assert (send[keep:cap] == 0).all() and send[cap, 0] == k_valid


def _nccl_gather_worker(rank, world, port, out):
    import os
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from pysilent_b200 import LineEndPipeline
    from pysilent_b200.distributed import PointGather, shard_range
    frames = np.stack([synthetic_frame(1, i, 480, 640) for i in range(5)])
    lo, hi = shard_range(len(frames), rank, world)
    pipe = LineEndPipeline(zoom_ratio=1.3)
    res = pipe.run_frames(torch.from_numpy(frames[lo:hi]).cuda())
    L = res.orient.shape[0] // (hi - lo)
    pts = torch.zeros((256, 4), dtype=torch.int64, device="cuda")
    pts[: len(res.points)] = res.points
    for native in (False, True):   # torch.distributed's collective, then the library's own silent_gather_points
        g = PointGather(256, L, torch.device("cuda", rank), native=native)
        got = None
        for _ in range(3):   # steady-state reuse of the slots
            got, counts = g.result(g.submit(pts, torch.tensor([len(res.points)], device="cuda"), lo))
        np.save(os.path.join(out, "nccl_%d_%d.npy" % (rank, native)), got.cpu().numpy())
        g.close()
    dist.destroy_process_group()


def test_point_gather_two_gpus_nccl(tmp_path):
    """Frames sharded over 2 GPUs, points gathered over NCCL: equal to the single-GPU run of the whole batch."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (gpurun --gpus 2)")
    import os
    import torch.multiprocessing as mp
    from pysilent_b200 import LineEndPipeline
    mp.spawn(_nccl_gather_worker, args=(2, 29600 + os.getpid() % 300, str(tmp_path)), nprocs=2, join=True)
    frames = np.stack([synthetic_frame(1, i, 480, 640) for i in range(5)])
    want = LineEndPipeline(zoom_ratio=1.3).run_frames(torch.from_numpy(frames).cuda()).points.cpu().numpy()
    for r in range(2):
        for native in (0, 1):
            assert np.array_equal(np.load(tmp_path / ("nccl_%d_%d.npy" % (r, native))), want), (r, native)


def test_outputs_stay_inside_their_buffers():
    """compute-sanitizer is not available on the GPU pool, so out-of-bounds WRITES of the bulk / staged stores are caught
    with canaries: every output lives in one arena between guard bands that must come back untouched (full tiles, ragged
    tiles, odd batch, a level width that is not a multiple of 4 = the non-bulk fallback)."""
    from pysilent_b200 import LineEndPipeline
    guard = 4096   # int64 words = 32 KB between tensors
    for (shape, center, scale, batch) in (((300, 420), (96, 64), 2 ** .5, 3), ((240, 330), (50, 36), 1.4, 2),
                                          ((1080, 1920), (288, 192), 2 ** .5, 5)):
        frames = np.stack([synthetic_frame(9, i, *shape) for i in range(batch)])
        pipe = LineEndPipeline(output_size=center, zoom_ratio=scale)
        dev = torch.from_numpy(frames).cuda()
        plan = pipe.plan_for(dev)
        n = batch * plan.levels
        elems = n * plan.h * plan.w * 3
        words_t = (elems * 4 + 7) // 8
        cap = 64 * n
        arena = torch.full((5 * guard + 2 * words_t + cap * 4 + 1,), 0x5A5A5A5A5A5A5A5A, dtype=torch.int64, device="cuda")
        off = guard
        orient = arena[off: off + words_t].view(torch.float32)[:elems].view(n, plan.h, plan.w, 3)
        off += words_t + guard
        line_end = arena[off: off + words_t].view(torch.float32)[:elems].view(n, plan.h, plan.w, 3)
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
        assert bool((arena[~used] == 0x5A5A5A5A5A5A5A5A).all()), "a kernel wrote outside its output tensors %s" % (shape,)
        ref = pipe.run_frames(dev)
        assert torch.equal(ref.orient.nan_to_num(-1.0), orient.nan_to_num(-1.0))
        assert torch.equal(ref.padded_line_end.nan_to_num(-1.0), line_end.nan_to_num(-1.0))
        assert torch.equal(ref.points, points[: int(count.item())])


def test_pipeline_four_channel_frames(c_oracle, default_filters):
    """BGRA frames (4 interleaved bytes per pixel, 3 colours used): the frame-pair pyramid kernel strides by the frame's
    channel count; equal to the 3-channel run of the same pixels and to the oracle."""
    from pysilent_b200 import LineEndPipeline
    bgr = np.stack([synthetic_frame(6, i, 360, 480) for i in range(3)])
    bgra = np.concatenate([bgr, np.full(bgr.shape[:3] + (1,), 255, np.uint8)], axis=-1)
    pipe = LineEndPipeline(output_size=(96, 64), zoom_ratio=1.5)
    want = pipe.run_frames(torch.from_numpy(bgr).cuda())
    got = pipe.run_frames(torch.from_numpy(bgra).cuda())
    assert torch.equal(got.orient.nan_to_num(-1.0), want.orient.nan_to_num(-1.0))
    assert torch.equal(got.padded_line_end.nan_to_num(-1.0), want.padded_line_end.nan_to_num(-1.0))
    assert torch.equal(got.points, want.points)
    pyr, ref = _oracle_pipeline(c_oracle, bgr, (96, 64), 1.5, default_filters)
    _check_stack(got, ref, None, "BGRA frames")
    host = pipe.run_host(bgra)
    assert np.array_equal(host.orient, ref["orient"], equal_nan=True) and np.array_equal(host.points, ref["points"])


def test_fused_stack_shape_sweep_bit_exact(c_oracle, default_filters):
    """Level shapes around every tile / vector boundary of the fused kernels (tile widths 48 and 64, tile heights 16 and
    32, runs of 8, 128-bit rows, bulk-store eligibility w % 4): values, NaN masks and gray bit-equal to the C oracle,
    including inputs with flat and dark patches (regulator pow path, 0 * inf)."""
    from pysilent_b200 import LineEndPipeline, _ops
    weights = LineEndPipeline().stack_weights()
    rs = np.random.RandomState(404)
    shapes = [(1, 1, 1), (1, 2, 3), (2, 7, 8), (1, 15, 47), (3, 16, 48), (1, 17, 49), (2, 31, 63), (1, 32, 64), (1, 33, 65),
              (2, 40, 96), (1, 48, 95), (1, 64, 100), (3, 35, 144), (1, 96, 130)]
    for n, h, w in shapes:
        x = (rs.rand(n, h, w, 3) * 255).astype(np.float32)
        if h > 8 and w > 8:
            x[0, : h // 3, : w // 2] = 37.0        # flat patch: blurred stripe response < 1 -> pow path
            x[-1, h // 2:, w // 2:] = 0.0          # dark patch: 0 * inf = NaN
        orient, line_end, gray = _ops.stack_fused(x, weights)
        ref = c_oracle.line_end_stack(x, default_filters)
        assert_bits(orient, ref["orient"], "orient %s" % ((n, h, w),))
        assert_bits(line_end, ref["padded"], "padded_line_end %s" % ((n, h, w),))
        assert_bits(gray, ref["gray"], "gray %s" % ((n, h, w),))


def test_pipeline_shape_sweep_bit_exact(c_oracle, default_filters):
    """Frame / level geometries around the fast-path conditions of the pipeline: frame rows that are (not) multiples of 16
    bytes (frame-pair pyramid kernel vs the per-pixel fallback), level widths that are (not) multiples of 4 / 48 / 64 / 72
    (bulk stores, tile choices), odd batches (a lone frame in the last pair), levels with unset tail rows. Device-resident
    and host-buffer calls, values and points bit-equal to the C oracle."""
    from pysilent_b200 import LineEndPipeline
    cases = [((97, 131), (24, 16), 2 ** .5, 3), ((120, 160), (72, 48), 1.3, 2), ((121, 163), (50, 34), 1.4, 1),
             ((200, 304), (76, 52), 1.5, 5), ((333, 448), (144, 96), 1.25, 2), ((480, 640), (100, 66), 1.7, 3)]
    for shape, center, scale, batch in cases:
        frames = np.stack([structured_frame(90 + i, *shape) if i % 2 else synthetic_frame(8, i, *shape) for i in range(batch)])
        pipe = LineEndPipeline(output_size=center, zoom_ratio=scale)
        pyr, ref = _oracle_pipeline(c_oracle, frames, center, scale, default_filters)
        res = pipe.run_frames(torch.from_numpy(frames).cuda())
        _check_stack(res, ref, None, "device %s" % (shape,))
        host = pipe.run_host(frames)
        _check_stack(host, ref, None, "host %s" % (shape,))


def test_orientation_bank_shape_sweep_bit_exact(c_oracle):
    """The fused bank path (config C4's kernels) around its tile boundaries: level widths that are (not) multiples of the
    32-pixel tile / the 4-pixel run / 4 floats, level heights that are (not) multiples of 16, odd batches, frames with flat
    and black patches (the regulator's slow path inside stack_bank_kernel). Values, NaN masks and points bit-equal to the
    oracle's bank composition."""
    from pysilent_b200 import LineEndPipeline
    cases = [((120, 160), (72, 48), 1.3, 2), ((200, 304), (76, 52), 1.5, 3), ((333, 448), (144, 96), 1.25, 1),
             ((480, 640), (100, 66), 1.7, 3), ((96, 128), (34, 18), 1.6, 5)]
    for shape, center, scale, batch in cases:
        frames = np.stack([structured_frame(60 + i, *shape) if i % 2 else synthetic_frame(9, i, *shape) for i in range(batch)])
        pipe = LineEndPipeline(output_size=center, zoom_ratio=scale, orientations=8)
        pyr = c_oracle.from_image(frames, 3, center, scale)
        ref = _oracle_bank(c_oracle, pyr, pipe.bank_filters(), (center[1] // 2, center[0] // 2))
        res = pipe.run_frames(torch.from_numpy(frames).cuda())
        assert tuple(res.orient.shape) == pyr.shape[:3] + (8,)
        _check_stack(res, ref, None, "bank %s" % (shape,))


def test_fused_stack_early_out_threshold_sweep(c_oracle, default_filters):
    """The regulator's early-out (quad sums prove blur > 1) around its own threshold: noise pyramids scaled so that the
    7x7 blur of the stripe sum sweeps from far below 1 (every gain != 1) through ~1 (mixed) to far above (every gain = 1).
    Bitwise against the oracle for every scale -- an unsound early-out would hand out a gain of exactly 1 where the
    reference's min(blur, 1) is below 1."""
    from pysilent_b200 import LineEndPipeline, _ops
    weights = LineEndPipeline().stack_weights()
    base = np.random.RandomState(77).rand(2, 40, 56, 3).astype(np.float32)
    mixed = 0
    for scale in (1e-5, 3e-5, 6e-5, 1e-4, 1.5e-4, 2e-4, 3e-4, 4e-4, 6e-4, 1e-3, 3e-3, 1e-2, 1.0, 30.0):
        x = (base * np.float32(scale * 255)).astype(np.float32)
        orient, line_end, gray = _ops.stack_fused(x, weights)
        ref = c_oracle.line_end_stack(x, default_filters)
        assert_bits(orient, ref["orient"], "orient, scale %g" % scale)
        assert_bits(line_end, ref["padded"], "padded_line_end, scale %g" % scale)
        gain_one = np.isclose(ref["orient"], ref["stripe"], rtol=0, atol=0) | (ref["stripe"] == 0)
        mixed += 0 < gain_one.mean() < 1
    assert mixed >= 3, "the sweep must cross the regime where only part of the gains are 1"


def test_pipeline_low_contrast_frames(c_oracle, default_filters):
    """uint8 frames with only a few grey levels: the blur of the stripe sum sits around 1, so the quick stack_b pass flags
    some tiles and not others and the fix-up pass redoes exactly those. Device and host entry points, bitwise."""
    from pysilent_b200 import LineEndPipeline
    pipe = LineEndPipeline(zoom_ratio=1.3)
    for levels_of_grey in (2, 3, 5, 9, 20):
        rs = np.random.RandomState(500 + levels_of_grey)
        frames = rs.randint(0, levels_of_grey, size=(3, 480, 640, 3)).astype(np.uint8)
        frames[1, 100:300, 200:500] = 1           # a flat patch inside the low-contrast noise
        pyr, ref = _oracle_pipeline(c_oracle, frames, (288, 192), 1.3, default_filters)
        res = pipe.run_frames(torch.from_numpy(frames).cuda())
        _check_stack(res, ref, None, "low contrast, %d grey levels" % levels_of_grey)
    host = pipe.run_host(frames)
    _check_stack(host, ref, None, "low contrast, host")


def _texture_alignment():
    """cudaDevAttrTextureAlignment of the current device, from the CUDA runtime torch has loaded (torch does not expose
    it): a linear texture's devPtr must be a multiple of it, so pyramid_pair_kernel reads other frame pointers by LDG."""
    import ctypes
    rt = ctypes.CDLL("libcudart.so.%s" % torch.version.cuda.split(".")[0])
    value = ctypes.c_int()
    assert rt.cudaDeviceGetAttribute(ctypes.byref(value), 14, torch.cuda.current_device()) == 0   # 14: TextureAlignment
    return value.value


def test_pyramid_texture_path_unaligned_frame_pointer(c_oracle, default_filters):
    """Frames handed over as a slice of a larger device buffer: the pointer is 16-byte aligned (required) but need not be
    aligned to the device's texture alignment. pyramid_pair_kernel reads frames at that alignment through the texture path
    and any others through its LDG variant, which is the same arithmetic; the code picks the route from the pointer.
     * a buffer at byte offset 16 (LDG), on a batch whose frames differ (texel indices of frame B) and that is odd (frame
       B = frame A in the last pair): bitwise equal to the run from an aligned buffer (texture) and to the oracle;
     * slices of a batch of 672000-byte frames: frame 1 starts off the alignment (LDG), frames 0 and 2 on it (texture);
     * 70 texture-aligned buffers, more than the plan's table of frame textures holds: the table is flushed (after a
       synchronisation) and refilled, and every result is the oracle's."""
    from pysilent_b200 import LineEndPipeline
    align = _texture_alignment()
    assert align > 16 and 672000 % align != 0, "the LDG cases below need a texture alignment above 16 bytes, got %d" % align
    frames = np.stack([synthetic_frame(2, i, 360, 640) for i in range(5)])
    dev = torch.from_numpy(frames).cuda()
    assert dev.data_ptr() % align == 0
    base = LineEndPipeline(zoom_ratio=1.5).run_frames(dev)
    buf = torch.zeros(frames.size + 16, dtype=torch.uint8, device="cuda")
    shifted = buf[16:].view(frames.shape)
    assert shifted.data_ptr() % align != 0
    shifted.copy_(dev)
    other = LineEndPipeline(zoom_ratio=1.5).run_frames(shifted)
    for name in ("orient", "padded_line_end"):
        a, b = getattr(base, name).cpu().numpy(), getattr(other, name).cpu().numpy()
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), "%s differs at byte offset 16" % name
    assert np.array_equal(base.points.cpu().numpy(), other.points.cpu().numpy())
    _, ref = _oracle_pipeline(c_oracle, frames, (288, 192), 1.5, default_filters)
    _check_stack(other, ref, None, "frames at byte offset 16")

    frames = np.stack([synthetic_frame(7, i, 2000, 112) for i in range(4)])
    dev = torch.from_numpy(frames).cuda()
    pipe = LineEndPipeline(zoom_ratio=1.5)
    for lo, hi in ((1, 3), (1, 4), (2, 4), (0, 4)):
        _, ref = _oracle_pipeline(c_oracle, frames[lo:hi], (288, 192), 1.5, default_filters)
        _check_stack(pipe.run_frames(dev[lo:hi]), ref, None, "frames[%d:%d]" % (lo, hi))
    small = np.stack([synthetic_frame(3, i, 96, 160) for i in range(2)])
    assert small.size % align == 0
    big = torch.zeros(70 * small.size, dtype=torch.uint8, device="cuda")
    _, ref = _oracle_pipeline(c_oracle, small, (32, 24), 1.5, default_filters)
    pipe2 = LineEndPipeline(output_size=(32, 24), zoom_ratio=1.5)
    for i in range(70):   # more distinct buffers than the table holds: it is flushed (after a synchronisation) and refilled
        view = big[i * small.size: (i + 1) * small.size].view(small.shape)
        assert view.data_ptr() % align == 0
        view.copy_(torch.from_numpy(small))
        res = pipe2.run_frames(view)
        if i in (0, 1, 63, 64, 65, 69):
            _check_stack(res, ref, None, "buffer %d" % i)
