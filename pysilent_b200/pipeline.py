"""``LineEndPipeline``: the fused hot path behind the interface of the reference's ``LineEndDisplayer``.

Reference: ``slam_recognition/recognition_testing.py:20-144``. ``compile()`` there builds, per pyramid shape, the graph
rgc -> rgby -> orientation -> end filter -> relu/clip -> border mask -> value -> region-max feature points; ``run()``
feeds one pyramid and fetches the result tensors; ``callback(frame, cam_id)`` is what the camera thread calls.
Here the graph is three CUDA kernels (pyramid, fused stack, point emit) behind ``libsilent_b200.so``; "compiling" is
building a plan (tap tables) per frame shape, cached like the reference caches its session per shape (``:108-118``).
"""
import collections
import ctypes
import math

import numpy as np
import torch

from . import _lib, _ops
from .constant_convolutions.center_surround import midget_rgc, rgby_3
from .constant_convolutions.edge_orientation_detector import rgb_2d_stripe_tensors
from .constant_convolutions.gaussian_blur.gaussian_blur import blur_tensor
from .constant_convolutions.oriented_end_detector import rgb_2d_end_tensors
from .util.zoom.from_image import PyramidPlan, image_to_zoom_tensor, zoom_frames_and_plan

def orientation_bank_filters(n_orient=8):
    """Filters of BASELINE config C4 (SURVEY 8(d)): ``n_orient`` orientations at ``k * 360 / n_orient`` degrees built
    with the reference's per-vector generators (``stripe_tensor`` ``stripe_tensor.py:21-70``, ``end_tensor``
    ``oriented_end_detector.py:13-55``, ``blur_tensor`` ``gaussian_blur.py:13-54``). The generators only build square
    channel maps, so the stripe bank is ``[3,3,n,n]`` sliced to its first 3 input channels (the rgby output feeds it)."""
    from .constant_convolutions.edge_orientation_detector.stripe_tensor import stripe_tensor
    from .constant_convolutions.oriented_end_detector import end_tensor
    vecs = [np.array([np.cos(k * 2 * np.pi / n_orient), np.sin(k * 2 * np.pi / n_orient)]) for k in range(n_orient)]
    eye = np.eye(n_orient)
    spread = [1, 1, 1] + [0] * (n_orient - 3)
    stripe = sum(stripe_tensor(v, spread, list(eye[k] * 4), spread, list(-eye[k] * 4)) for k, v in enumerate(vecs))
    end = sum(end_tensor(3 * v, list(eye[k]), list(.25 * eye[k]), list(eye[k]), list(.5 * eye[k]))
              for k, v in enumerate(vecs))
    return dict(rgc=midget_rgc(2), rgby=rgby_3(2), stripe=np.ascontiguousarray(stripe[:, :, :3, :]),
                blur=blur_tensor(2, 7, channels_in=n_orient, channels_out=n_orient), end=end)


def host_round_trip(staged, device, run, pinned):
    """``run`` on a copy of the page-locked host tensor ``staged`` on ``device``; returns the tensors it returns as numpy
    arrays. The upload and every download are asynchronous, result i into the page-locked ``pinned(i, shape, dtype)``,
    and the stream is synchronised once for all of them."""
    with torch.cuda.device(device):
        outs = []
        for i, t in enumerate(run(staged.to(device, non_blocking=True))):
            host = pinned(i, tuple(t.shape), t.dtype)
            host.copy_(t, non_blocking=True)
            outs.append(host.numpy())
        torch.cuda.current_stream().synchronize()
    return outs


# defaults of run_frames_motion / run_host_motion (profiles/motion_bench_b200.json)
MOTION_THRESHOLD = 2.0   # frame pixels
MOTION_HYPOTHESES = 256

# routes of frames (LineEndPipeline._frame_route)
PLAN, CONVERT, PYRAMID = "plan", "convert", "pyramid"

LineEndResult = collections.namedtuple("LineEndResult", "orient padded_line_end gray points")
LineEndResult.__doc__ = """orient: ``orient_tensor`` [N,h,w,3]; padded_line_end: ``padded_line_end_tensor`` [N,h,w,3];
gray: ``gray_line_end_tensor`` [N,h,w,1] (or None); points: int64 [K,4] rows (level, y, x, 0) (``top_percent_points``)."""

PointRecords = collections.namedtuple("PointRecords", "points frame_offsets frame_yx gray orient line_end")
PointRecords.__doc__ = """The feature points of a batch of B frames with what fired at each (``silent_point_records``):
points: int64 [K,4] rows (level, y, x, 0) as ``LineEndResult.points``, level = frame * L + l; frame_offsets: int64
[B+1], the rows of frame b are ``points[frame_offsets[b]:frame_offsets[b + 1]]``; frame_yx: float32 [K,2], the
point's (row, column) in its frame, ``y0 + y * (n_in - 1) / (n_out - 1)`` per axis (``PyramidPlan.level_coords``; NaN
on an axis the level defines as 0); gray: float32 [K], orient and line_end: float32 [K,C], the values of ``gray``,
``orient`` and ``padded_line_end`` at the point (float16 outputs widened exactly).

With a patch radius r (``patch_radius=r`` of ``run_frames_records`` / ``run_host_records``, ``silent_point_patches``)
gray is float32 [K,P,P], orient and line_end float32 [K,P,P,C], P = 2r + 1: the values at pixel (y + dy, x + dx) of the
point's level, dy and dx in [-r, r], at [r + dy, r + dx]; +0.0 where that pixel leaves the level (what the stack's
SAME zero padding reads there). points, frame_offsets and frame_yx stay one per point. gray, orient and line_end are
views of one float32 values tensor [K,1 + 2C] ([K,P,P,1 + 2C] with a patch)."""

PointMatches = collections.namedtuple("PointMatches", "next prev distance")
PointMatches.__doc__ = """Links between the feature points of consecutive frames of one batch (``silent_match_points``),
over the K rows of the ``PointRecords`` they come with: next: int64 [K], the row j of frame f + 1 that row i of frame f
matches, or -1; prev: int64 [K], the row i for that j, or -1; distance: float32 [K], SSD(i, next[i]), or NaN where next
is -1. next and prev are consistent (``prev[next[i]] == i``), so following next gives a track through the batch.

Level n of frame f (n = f * L + l) pairs with level n + L of frame f + 1. The candidates of row i in the next frame are
the rows j of that level with |y_j - y_i| <= R and |x_j - x_i| <= R in level pixels (R = ``search_radius``); in the
previous frame the same with n - L. The distance of two rows is the float32 SSD of their descriptors, the record's
values flattened (E = P * P * (1 + 2C) with a patch, 1 + 2C without), in a fixed order: lane k = 0..31 sums
``d = a_e - b_e; s_k = s_k + d * d`` over e = k, k + 32, ... from +0.0, then ``s_k = s_k + s_(k xor m)`` for m = 16, 8, 4,
2, 1 gives SSD = s_0; every operation rounded to nearest, no fused products, symmetric in the two rows bit for bit. A
candidate of NaN SSD is ignored, so a row of NaN values matches nothing. In each direction d1 is the smallest SSD over
the candidates (ties to the smaller row) and d2 the smallest over the others (+inf without any); the best candidate is
the raw link iff ``d1 <= float32(max_ratio) * d2`` (rounded). ``max_ratio`` = 1 turns the test off; it applies to SSD,
so Lowe's 0.8 on distances is 0.64 here. i -> j is accepted iff j is i's raw link in the next frame and i is j's in the
previous one. Rows of the last frame have next = -1 and rows of frame 0 prev = -1: matches never span calls, so a stream
processed in batches keeps one frame of overlap between consecutive batches to link them."""

PointMotion = collections.namedtuple("PointMotion", "transform inlier_count matched inlier")
PointMotion.__doc__ = """How the camera moved between consecutive frames of one batch, and which matches agree with that
motion (``silent_estimate_motion``), over the B frames and K rows of the ``PointRecords`` and ``PointMatches`` it comes
with: transform: float64 [B - 1, 2, 3], per pair (f, f + 1) the affine map T with ``[y1, x1] = T[:, :2] @ [y0, x0] +
T[:, 2]`` in frame pixels, (y, x) order as ``frame_yx``; all NaN when the pair has fewer than 3 correspondences or every
hypothesis is degenerate; inlier_count: int64 [B - 1], the correspondences T keeps (0 then); matched: int64 [B - 1], the
pair's correspondences M_f; inlier: uint8 [K], 1 iff the row is a correspondence of its pair and an inlier of T.

The correspondences of pair f are the rows i of frame f (``frame_offsets[f] <= i < frame_offsets[f + 1]``), in row
order, with ``next[i] >= 0`` and ``frame_yx[i]``, ``frame_yx[next[i]]`` all finite (rows of a level that defines an axis
as 0 have NaN coordinates and never take part): c_k = (y0, x0, y1, x1), k = 0 .. M_f - 1.

Hypothesis h = 0 .. H - 1 (H = ``hypotheses``) draws k_d = mulhi64(u_d, M_f), d = 0, 1, 2, with u_d =
splitmix64(seed ^ splitmix64((f << 32) | (h << 2) | d)) (Vigna's splitmix64 finaliser with its 0x9e3779b97f4a7c15
increment, 64-bit wrapping). It is degenerate if two draws are equal. Otherwise, in float64: with (y0, x0) the source of
c_k0 and dyj = yj - y0, dxj = xj - x0 for the sources of c_k1, c_k2, D = dy1 * dx2 - dx1 * dy2, degenerate if
``!(|D| >= 1)``; per target u (y1, then x1): du1 = u_k1 - u_k0, du2 = u_k2 - u_k0, a = (du1 * dx2 - dx1 * du2) / D,
b = (dy1 * du2 - du1 * dy2) / D, c = u_k0 - (a * y0 + b * x0).

A model T scores in float32: m = float32(T), rounded once; c_k is an inlier iff ``e_y * e_y + e_x * e_x <= t * t`` with
t = float32(threshold), ``e_y = y1 - ((m_a * y0 + m_b * x0) + m_c)`` and e_x likewise, every operation rounded, no fused
products. The best hypothesis has the most inliers, ties to the smaller h.

Refit: one least-squares step on the inliers of the best hypothesis. With (py, px, qy, qx) = its c_k0 and Y = y0 - py,
X = x0 - px, U = y1 - qy, V = x1 - qx in float64, the 11 sums of Y, X, YY, YX, XX, U, YU, XU, V, YV, XV are each taken in
a fixed order: thread t = 0..255 adds its terms over k = t, t + 256, ... from +0.0; within each warp of 32 threads
``s_t = s_t + s_(t xor b)`` for b = 16, 8, 4, 2, 1; the 8 warps' lane-0 sums w are added as ((w_0 + w_1) + ...) + w_7.
The two 3 x 3 normal systems are solved by their adjugate (``silent_estimate_motion`` in ``silent_b200.h`` spells out
every operation) and the translation is moved back by ``c = (q + c') - (a * py + b * px)``. The refit is kept if its six
values are finite and it scores at least as many inliers; otherwise the best hypothesis's T is.

Matches never span calls, so motion never does either; one frame (B = 1) gives empty pair outputs and inlier all 0."""


class LineEndPipeline:
    """Drop-in for the compute half of ``LineEndDisplayer`` (camera / window handling is out of scope).

    Constructor keywords follow ``PyramidDisplayer.__init__`` (``pyramid_displayer.py:22``): ``output_size`` is
    ``(w, h)`` of every pyramid level, ``zoom_ratio`` the scale between levels.

    ``out_dtype`` is the dtype of ``orient`` and ``padded_line_end`` on every entry point: ``torch.float32`` (default) or
    ``torch.float16``. With float16 each value is the float32 result rounded once to nearest even, as ``.half()`` rounds
    it; the fused kernels store it that way (half the output bytes, on the device and over the host link), the other
    paths cast their float32 result once. ``gray`` stays float32, and the feature points are the float32 call's.

    ``frame_format`` is the layout of the frames every entry point takes: ``"bgr"`` (default), ``[H, W, 3]`` per frame,
    or ``"nv12"``, the 4:2:0 layout video decoders produce: one uint8 ``[H * 3 / 2, W]`` array per frame (H rows of Y,
    then H / 2 rows of interleaved U, V), H and W even. An NV12 call returns exactly what the same call returns on the
    frames ``cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12)`` makes of them; the conversion runs on the GPU, in front of the
    pyramid, and only the bytes of the NV12 frames cross the host link.

    ``peaks`` chooses the feature points of every entry point. ``None`` (default) keeps the reference's region maxima
    (``max_value_indices_region``, one to four points per level). A real number p in [0, 1] emits the peaks of every
    level instead (``silent_peak_points``): each pixel that is > 0, >= the level's top-percent threshold
    ``float32(1 - p) * max + float32(p) * min`` (``top_value_points``) and >= every pixel of its 3 x 3 neighbourhood. A
    plateau fires on every pixel, and a level holding a NaN or only zeros emits nothing. The rows keep the format and
    order of the region maxima, so records, patches and the point gathers take them as they are.
    """

    def __init__(self, n_dimensions=2, output_size=(288, 192), output_colors=3, zoom_ratio=math.e ** .5, device=None,
                 orientations=None, out_dtype=torch.float32, frame_format="bgr", peaks=None):
        self.peaks = _ops.peak_percent(peaks) if peaks is not None else None
        if out_dtype not in _ops.OUT_DTYPES:
            raise ValueError("out_dtype must be torch.float32 or torch.float16, got %r" % (out_dtype,))
        if not isinstance(frame_format, str) or frame_format not in _ops.FRAME_FORMATS:
            raise ValueError("frame_format must be one of %s, got %r" % (", ".join(_ops.FRAME_FORMATS), frame_format))
        self.out_dtype = out_dtype
        self.frame_format = frame_format
        # None: the reference's 3 simplex orientations; n: a bank of n orientations (config C4: 8). Fused kernels for n = 4,
        # 8, 12 and 16; other n up to 8 run operator by operator
        self.orientations = orientations
        self._bank = None
        self._bank_weights = None
        self.output_size = tuple(output_size)
        self.output_colors = output_colors
        self.zoom_ratio = zoom_ratio
        self.simplex_end_stop = rgb_2d_end_tensors()                                   # recognition_testing.py:29
        self.region_shape = [1, self.output_size[1] / 2.0, self.output_size[0] / 2.0, self.output_colors]   # :40
        self.blur_size = 7
        self.device = torch.device(device) if device is not None else None
        self._weights = None
        self._weights_key = None
        self._plans = {}   # per instance: a plan owns workspace buffers, so pipelines (cameras, threads) never share one

    # -- weights ------------------------------------------------------------------------------------------------------
    def filters(self):
        """HWIO float64 filters in graph order (recognition_testing.py:69-73)."""
        return dict(rgc=midget_rgc(2), rgby=rgby_3(2), stripe=rgb_2d_stripe_tensors(),
                    blur=blur_tensor(2, lengths=self.blur_size), end=np.asarray(self.simplex_end_stop))

    def stack_weights(self):
        end = np.ascontiguousarray(np.asarray(self.simplex_end_stop), dtype=np.float32)
        key = (end.tobytes(), self.blur_size)
        if self._weights is None or key != self._weights_key:
            f = self.filters()
            self._weights = _lib.make_stack_weights(f["rgc"], f["rgby"], f["stripe"], f["blur"], f["end"])
            self._weights_key = key
        return self._weights

    def _device(self):
        _ops._require_cuda()
        return self.device if self.device is not None else torch.device("cuda", torch.cuda.current_device())

    def _half(self):
        return self.out_dtype == torch.float16

    def _nv12(self):
        return self.frame_format == "nv12"

    def _points(self, gray):
        """Feature points of ``gray``: the maxima of the reference's region windows (``recognition_testing.py:40``), or
        its peaks with ``peaks`` set."""
        if self.peaks is not None:
            return _ops.peak_points(gray, self.peaks)
        rh, rw = self.region_shape[1], self.region_shape[2]
        if int(rh) != rh or int(rw) != rw:
            raise ValueError("Ambiguous dimension: %s" % ([rh, rw],))
        return _ops.max_value_indices_region(gray, int(rh), int(rw))

    # -- graph on a pyramid (LineEndDisplayer.run) --------------------------------------------------------------------
    def run(self, pyramid_tensor, want_points=True):
        """S1-S8 on a pyramid ``[N, h, w, 3]`` (numpy or CUDA tensor). One fused kernel + the emit kernels."""
        if self.orientations is not None:
            return self.run_bank(pyramid_tensor, want_points)
        return self._run_pyramid(pyramid_tensor, None, want_points)

    def run_unfused(self, pyramid_tensor, want_points=True):
        """The same graph through the per-operator kernels (any filter structure, any blur size)."""
        return self._run_operators(pyramid_tensor, self.filters, want_points)

    def run_bank(self, pyramid_tensor, want_points=True):
        """Config C4: S1-S2 on 3 channels, S3-S7 on an ``orientations``-channel bank (same composition as ``compile()``,
        ``recognition_testing.py:69-77``), on the route ``_run_pyramid`` gives."""
        return self._run_pyramid(pyramid_tensor, self._bank_width(), want_points)

    def _run_pyramid(self, pyramid_tensor, nb, want_points):
        """``run`` and ``run_bank`` with ``nb`` orientations (None: the reference's three). A finite pyramid goes through
        the fused stack without a bank at blur size 7 (``silent_stack_fused``), and through the fused bank stack with 12
        or 16 orientations (``silent_stack_bank``; a non-finite one raises ValueError). All else goes operator by
        operator, banks of 4 and 8 included: their results are pinned to the operators' order, not the fused one."""
        fused = self.blur_size == 7 if nb is None else nb > 8
        if not fused:
            return self._run_operators(pyramid_tensor, self.filters if nb is None else self.bank_filters, want_points)
        x = _ops.as_device_tensor(pyramid_tensor)
        # the fused kernels skip exact-zero weights and shortcut the regulator where the blur is provably >= 1: valid for
        # finite input only (include/silent_b200.h). NaN / Inf / huge values go operator by operator, like the graph.
        if not _ops.fused_input_ok(x):
            if nb is not None:
                raise ValueError("a pyramid with NaN, Inf or values beyond 1e30 goes operator by operator, which "
                                 "supports at most 8 orientations (got %d)" % nb)
            return self._run_operators(x, self.filters, want_points)
        if nb is None:
            orient, line_end, gray = _ops.stack_fused(x, self.stack_weights(), out_dtype=self.out_dtype)
        else:
            orient, line_end, gray = _ops.stack_bank(x, self.orientation_bank(), out_dtype=self.out_dtype)
        return LineEndResult(orient, line_end, gray, self._points(gray) if want_points else None)

    def _run_operators(self, pyramid_tensor, filters, want_points):
        """The graph of ``compile()`` (``recognition_testing.py:69-77``) one operator kernel at a time, on the HWIO
        filters ``filters()`` returns (``self.filters`` or ``self.bank_filters``)."""
        x = _ops.as_device_tensor(pyramid_tensor)
        f = filters()
        x = _ops.conv2d(_ops.conv2d(x, f["rgc"], post=_lib.POST_RELU), f["rgby"], post=_lib.POST_RELU)
        orient = _ops.regulate(_ops.conv2d(x, f["stripe"], post=_lib.POST_RELU), f["blur"], 1.0, .1)
        line_end = _ops.conv2d(orient, f["end"], post=_lib.POST_RELU_CLIP, clip_max=255.0)
        padded = _ops.pad_inwards(line_end, 2, 2, 2, 2)
        gray = _ops.value_from_color(padded)
        points = self._points(gray) if want_points else None
        if self._half():   # the float32 result in out_dtype: orient and padded_line_end rounded once, gray and points kept
            orient, padded = orient.half(), padded.half()
        return LineEndResult(orient, padded, gray, points)

    def bank_filters(self):
        if self._bank is None:
            self._bank = orientation_bank_filters(self.orientations)
        return self._bank

    def _bank_width(self):
        """``orientations``, after rejecting the widths no path runs (before anything touches the GPU)."""
        nb = int(self.orientations)
        if nb > 16 or (nb > 8 and nb % 4):
            raise ValueError("orientations=%d is not supported: a bank has up to 8 orientations, or 12 or 16 (fused "
                             "kernels exist for 4, 8, 12 and 16)" % nb)
        return nb

    def orientation_bank(self):
        """The bank's filters packed for the fused kernels (``silent_orientation_bank``)."""
        if self._bank_weights is None:
            f = self.bank_filters()
            self._bank_weights = _lib.make_orientation_bank(f["rgc"], f["rgby"], f["stripe"], f["blur"], f["end"])
        return self._bank_weights

    # -- frames resident in HBM ---------------------------------------------------------------------------------------
    def _plan(self, frame_shape, frame_dtype, device, frame_format="bgr"):
        """Plan cache keyed like the reference's per-shape session (``recognition_testing.py:108-118``). The cache is
        per pipeline: use one ``LineEndPipeline`` per camera thread, as the reference uses one displayer per camera.
        NV12 plans take ``frame_shape`` ``(H, W, 3)`` of the image."""
        key = (tuple(int(v) for v in frame_shape), frame_dtype, frame_format, self.output_colors, self.output_size,
               float(self.zoom_ratio), str(device))
        plan = self._plans.get(key)
        if plan is None:
            with torch.cuda.device(device):
                plan = PyramidPlan(frame_shape, frame_dtype, self.output_colors, self.output_size, self.zoom_ratio,
                                   frame_format)
            self._plans[key] = plan
        return plan

    def plan_for(self, frames):
        """The plan of a batch of frames in the pipeline's ``frame_format``."""
        if self._nv12():
            h, w = _ops.nv12_frame_hw(frames.shape, frames.dtype)
            return self._plan((h, w, 3), torch.uint8, frames.device, "nv12")
        return self._plan(frames.shape[1:], frames.dtype, frames.device)

    def _frame_route(self, nb, frame_format, dtype, frame_shape):
        """How ``run_frames`` and ``run_host`` compute on frames of ``frame_format``, torch ``dtype`` and a shape ending
        in ``[W, C]`` (NV12: ``[W]``) with ``nb`` orientations (None: the reference's three):
        - ``PLAN``: a plan of the frames' format and the fused pipeline, ``silent_pipeline_run[_f16]`` (a bank:
          ``silent_pipeline_run_orientations[_f16]``);
        - ``CONVERT``: ``_ops.nv12_to_bgr``, then the route of the BGR frames;
        - ``PYRAMID``: ``image_to_zoom_tensor``, then ``run_bank``.

        BGR frames without a bank take ``PLAN``; with a bank they take it where the fused bank kernels serve them, else
        ``PYRAMID``. NV12 frames take ``PLAN`` where the BGR frames they convert to would, with blur size 7 and
        ``output_colors`` 3; else ``CONVERT``. Quirks kept as they are:
        - ``PYRAMID`` ignores ``out=`` and ``points_capacity``: it returns new tensors, ``gray`` and every point;
        - on ``PYRAMID`` a bank of 12 or 16 raises ValueError for non-finite frames, and a bank of 4 or 8 runs operator
          by operator, in the operators' order;
        - a blur size other than 7 sends a bank to ``PYRAMID``, though a bank's filters blur with 7 taps at any size;
        - without a bank, a blur size other than 7 raises in ``make_stack_weights`` and ``output_colors`` other than 3
          in the C argument check, on NV12 frames after ``CONVERT``."""
        fusable = self.blur_size == 7 and self.output_colors == 3
        if frame_format == "nv12":   # the BGR frames they convert to are uint8 [.., W, 3]
            return PLAN if fusable and self._frame_route(nb, "bgr", torch.uint8, (frame_shape[-1], 3)) == PLAN else CONVERT
        w, c = frame_shape[-2:]
        # a bank's pyramid is the frame-pair kernel, which reads rows of whole 16-byte words of uint8 frames (the C
        # condition is pyramid_pair_supported, csrc/pyramid.cu)
        if nb is None or (nb in _lib.FUSED_BANK_WIDTHS and dtype == torch.uint8 and c >= 3 and fusable
                          and (w * c) % 16 == 0):
            return PLAN
        return PYRAMID

    def run_frames(self, frames, want_points=True, points_capacity=None, out=None):
        """frames: CUDA ``[B, H, W, 3]`` uint8/float32 (``frame_format="nv12"``: ``[B, H * 3 / 2, W]`` uint8) ->
        LineEndResult over ``B * L`` levels (pyramid + S1-S8). A single frame may come without its batch axis.

        ``out`` may carry preallocated ``(orient, padded_line_end, points, count)`` tensors to avoid allocation in a
        steady-state loop; ``points`` then holds ``count`` valid rows (no host sync is performed in that case). With
        ``orientations`` set, orient and padded_line_end have ``orientations`` channels instead of 3. Both are of
        ``out_dtype``, and so must be the ``out`` buffers.
        """
        nb = self._bank_width() if self.orientations is not None else None
        if out is not None and (out[0].dtype != self.out_dtype or out[1].dtype != self.out_dtype):
            raise ValueError("run_frames(out=...) needs orient and padded_line_end buffers of %s, got %s and %s"
                             % (self.out_dtype, out[0].dtype, out[1].dtype))
        nv12_hw = _ops.nv12_frame_hw(frames.shape, frames.dtype) if self._nv12() else None
        frames = (frames if frames.dim() == (3 if nv12_hw else 4) else frames.unsqueeze(0)).contiguous()
        route = self._frame_route(nb, self.frame_format, frames.dtype, frames.shape)
        if route == CONVERT:
            frames, nv12_hw = _ops.nv12_to_bgr(frames), None
            route = self._frame_route(nb, "bgr", frames.dtype, frames.shape)
        if route == PYRAMID:
            return self.run_bank(image_to_zoom_tensor(frames, self.output_colors, self.output_size, self.zoom_ratio),
                                 want_points)
        return self._run_plan(frames, nb, want_points, points_capacity, out, nv12_hw)

    def _plan_of(self, frames, nv12_hw):
        """The plan of a contiguous batch on the ``PLAN`` route (see ``_run_plan``)."""
        if nv12_hw is None:
            return self._plan(frames.shape[1:], frames.dtype, frames.device)
        return self._plan(nv12_hw + (3,), torch.uint8, frames.device, "nv12")

    def _run_plan(self, frames, nb, want_points, points_capacity, out, nv12_hw):
        """The ``PLAN`` route on a contiguous batch: BGR / float ``[B, H, W, C]``, or NV12 ``[B, H * 3 / 2, W]`` of an
        ``nv12_hw`` = ``(H, W)`` image."""
        plan = self._plan_of(frames, nv12_hw)
        b = int(frames.shape[0])
        plan.reserve(b)
        n = b * plan.levels
        dev = frames.device
        if out is None:
            orient = torch.empty((n, plan.h, plan.w, nb or 3), dtype=self.out_dtype, device=dev)
            line_end = torch.empty_like(orient)
            cap = int(points_capacity) if points_capacity else max(64 * n, 1024)
            points = torch.empty((cap, 4), dtype=torch.int64, device=dev)
            count = torch.zeros(1, dtype=torch.int64, device=dev)
        else:
            orient, line_end, points, count = out
            cap = int(points.shape[0])
        # the 3-orientation stack (silent_pipeline_run, no pyramid output) or the fused bank (config C4 and its variants:
        # pyramid_pair_kernel -> stack_a -> stack_bank_kernel -> emit)
        if nb is None:
            name, args = "silent_pipeline_run", (ctypes.byref(self.stack_weights()), _ops.ptr(frames), b, None)
        else:
            name, args = "silent_pipeline_run_orientations", (ctypes.byref(self.orientation_bank()), _ops.ptr(frames), b)
        if self._half():
            name += "_f16"
        # the emit step: the region maxima inside the pipeline call, or the peaks after it on the plan's own gray
        peaks = want_points and self.peaks is not None
        with torch.cuda.device(dev):
            _lib.check(getattr(_lib.lib(), name)(
                plan.handle, *args, _ops.ptr(orient), _ops.ptr(line_end), _ops.ptr(points), cap,
                _ops.ptr(count) if want_points and not peaks else None, _ops.stream_ptr()), name)
        if peaks:
            _ops.plan_peak_points(plan, b, self.peaks, points, count)
        if out is not None:
            return LineEndResult(orient, line_end, None, points)
        if not want_points:
            return LineEndResult(orient, line_end, None, None)
        total = int(count.item())
        if total > cap and peaks:   # only the emit again, on the plan's gray of this call
            points = self._plan_peaks(plan, b, total, count)
        elif total > cap:   # rare (e.g. an all-black level emits every pixel): redo the emit with room for everything
            return self._run_plan(frames, nb, want_points, total, None, nv12_hw)
        return LineEndResult(orient, line_end, None, points[:total])

    def _plan_peaks(self, plan, b, capacity, count):
        """The peaks of the plan's gray of its latest call (``b`` frames) into new points of ``capacity`` rows."""
        points = torch.empty((capacity, 4), dtype=torch.int64, device=count.device)
        _ops.plan_peak_points(plan, b, self.peaks, points, count)
        return points

    # -- feature-point records ------------------------------------------------------------------------------------------
    def run_frames_records(self, frames, points_capacity=None, out=None, patch_radius=None):
        """``run_frames`` on the same frames and route, returning the feature points with their frame coordinates and
        the responses at each (``PointRecords`` of CUDA tensors) instead of the whole output tensors.

        ``out`` may carry preallocated ``(orient, padded_line_end, points, count, frame_offsets, frame_yx, values)``
        buffers: the first four as for ``run_frames(out=...)``, then int64 ``[B + 1]``, float32 ``[capacity, 2]`` and
        float32 ``[capacity, 1 + 2 * C]`` (C = 3 or ``orientations``). No host synchronisation is performed then, and
        the result's tensors are views of those buffers over the whole capacity: the first ``min(count, capacity)`` rows
        are written and ``frame_offsets`` counts only those. Without ``out`` the call synchronises once to trim to the
        points found, and redoes the call with room for all of them when they exceed ``points_capacity``.

        With an int ``patch_radius`` r in [0, 31] each record carries the patch of side P = 2r + 1 around its point
        (see ``PointRecords``); ``out``'s ``values`` is then float32 ``[capacity, P, P, 1 + 2 * C]``. Without ``out``
        the call synchronises once on the count first and sizes the patches by the points found, not by the capacity.

        The records are those of every route ``run_frames`` takes; like there, the ``PYRAMID`` route ignores ``out`` and
        ``points_capacity`` and returns every point in new tensors. Banks of widths other than 4, 8, 12 and 16, and a
        ``patch_radius`` that is not an int in [0, 31], raise ValueError."""
        return self._records(*self._record_rows(frames, points_capacity, out, patch_radius)[1])

    def _record_rows(self, frames, points_capacity, out, radius=None):
        """``run_frames_records`` as ``(L, (points, frame_offsets, frame_yx, values [K, 1 + 2C] or [K, P, P, 1 + 2C]))``,
        L the levels per frame of the route's plan."""
        radius = _ops.patch_radius(radius)
        nb = self._bank_width() if self.orientations is not None else None
        c = nb or 3
        if c not in _lib.RECORD_CHANNELS:
            raise ValueError("feature-point records need 3 orientations or a bank of 4, 8, 12 or 16, got %d" % c)
        if points_capacity is not None and int(points_capacity) < 0:
            raise ValueError("points_capacity must be >= 0, got %d" % int(points_capacity))
        if out is not None:
            if len(out) != 7:
                raise ValueError("run_frames_records(out=...) takes (orient, padded_line_end, points, count, "
                                 "frame_offsets, frame_yx, values), got %d buffers" % len(out))
            if out[0].dtype != self.out_dtype or out[1].dtype != self.out_dtype:
                raise ValueError("run_frames_records(out=...) needs orient and padded_line_end buffers of %s, got %s "
                                 "and %s" % (self.out_dtype, out[0].dtype, out[1].dtype))
        nv12_hw = _ops.nv12_frame_hw(frames.shape, frames.dtype) if self._nv12() else None
        frames = (frames if frames.dim() == (3 if nv12_hw else 4) else frames.unsqueeze(0)).contiguous()
        if out is not None and radius is not None:
            _ops.check_record_buffers(int(frames.shape[0]), int(out[2].shape[0]), c, radius, *out[4:])
        route = self._frame_route(nb, self.frame_format, frames.dtype, frames.shape)
        if route == CONVERT:
            frames, nv12_hw = _ops.nv12_to_bgr(frames), None
            route = self._frame_route(nb, "bgr", frames.dtype, frames.shape)
        if route == PYRAMID:
            zframes, zplan = zoom_frames_and_plan(frames, self.output_colors, self.output_size, self.zoom_ratio)
            res = self.run_bank(zplan.build(zframes), True)
            count = torch.full((1,), len(res.points), dtype=torch.int64, device=res.points.device)
            recs = _ops.point_records(zplan, zframes.shape[0], res.points, count, res.orient, res.padded_line_end,
                                      res.gray, radius=radius)
            return zplan.levels, (res.points,) + recs
        levels = self._plan_of(frames, nv12_hw).levels
        return levels, self._run_plan_records(frames, nb, points_capacity, out, nv12_hw, radius)

    def _run_plan_records(self, frames, nb, points_capacity, out, nv12_hw, radius=None):
        plan = self._plan_of(frames, nv12_hw)
        b = int(frames.shape[0])
        if out is None:
            dev = frames.device
            cap = int(points_capacity) if points_capacity is not None else max(64 * b * plan.levels, 1024)
            orient = torch.empty((b * plan.levels, plan.h, plan.w, nb or 3), dtype=self.out_dtype, device=dev)
            run_out = (orient, torch.empty_like(orient), torch.empty((cap, 4), dtype=torch.int64, device=dev),
                       torch.zeros(1, dtype=torch.int64, device=dev))
            bufs = (None, None, None)
        else:
            run_out, bufs = tuple(out[:4]), tuple(out[4:])
        orient, line_end, points, count = run_out
        self._run_plan(frames, nb, True, None, run_out, nv12_hw)
        # gray: the plan's own, written by the call above on this stream
        if out is None and radius is not None:
            # patches for the whole default capacity could take GBs: size them by the points found
            total = int(count.item())
            if total > points.shape[0] and self.peaks is not None:   # only the emit again, as run_frames
                points = self._plan_peaks(plan, b, total, count)
            elif total > points.shape[0]:
                return self._run_plan_records(frames, nb, total, None, nv12_hw, radius)
            points = points[:total]
            return (points,) + _ops.point_records(plan, b, points, count, orient, line_end, None, radius=radius)
        recs = _ops.point_records(plan, b, points, count, orient, line_end, None, *bufs, radius=radius)
        if out is not None:
            return (points,) + recs
        total = int(count.item())
        if total > points.shape[0] and self.peaks is not None:   # only the emit again, then the records of every point
            points = self._plan_peaks(plan, b, total, count)
            recs = _ops.point_records(plan, b, points, count, orient, line_end, None)
        elif total > points.shape[0]:   # as run_frames: redo with room for every point
            return self._run_plan_records(frames, nb, total, None, nv12_hw)
        frame_offsets, frame_yx, values = recs
        return points[:total], frame_offsets, frame_yx[:total], values[:total]

    @staticmethod
    def _records(points, frame_offsets, frame_yx, values):
        """``PointRecords`` of the rows ``_record_rows`` returns (gray, orient and line_end are views of ``values``)."""
        c = (values.shape[-1] - 1) // 2
        return PointRecords(points, frame_offsets, frame_yx, values[..., 0], values[..., 1:1 + c], values[..., 1 + c:])

    def run_host_records(self, frames, points_capacity=4096, patch_radius=None):
        """``run_frames_records`` on host frames: numpy ``[B, H, W, 3]`` (``frame_format="nv12"``: ``[B, H * 3 / 2, W]``
        uint8), pageable or page-locked. The frames go up once and only the records come back (``PointRecords`` of
        numpy arrays): ``orient`` and ``padded_line_end`` never cross the host link. ``points_capacity`` sizes the first
        attempt; every point is returned. ``patch_radius`` as for ``run_frames_records`` (checked before the upload)."""
        radius = _ops.patch_radius(patch_radius)
        staged, dev = self._stage_host(frames)
        rows = host_round_trip(staged, dev, lambda x: self._record_rows(x, points_capacity, None, radius)[1],
                               lambda i, shape, dtype: torch.empty(shape, dtype=dtype, pin_memory=True))
        return self._records(*rows)

    def _stage_host(self, frames):
        """Host frames of ``run_host_records`` / ``run_host_matches`` as a batched page-locked tensor, and the device."""
        frames = np.asarray(frames)
        nv12_hw = _ops.nv12_frame_hw(frames.shape, frames.dtype) if self._nv12() else None
        frames = np.ascontiguousarray(frames)
        if frames.ndim == (2 if nv12_hw else 3):
            frames = frames[np.newaxis]
        if frames.dtype != np.uint8:
            frames = frames.astype(np.float32)
        dev = self._device()
        staged = torch.from_numpy(frames)
        if not staged.is_pinned():   # page-locked frames (e.g. views of pinned tensors) go up in place
            staged = staged.pin_memory()
        return staged, dev

    # -- feature-point matches ------------------------------------------------------------------------------------------
    def run_frames_matches(self, frames, patch_radius, search_radius, max_ratio=1.0, points_capacity=None):
        """The records of ``run_frames_records(frames, points_capacity, patch_radius=patch_radius)`` and the links between
        the points of consecutive frames (``PointRecords``, ``PointMatches``), all CUDA tensors. Each point's descriptor
        is its record's values: the patch of radius ``patch_radius`` (an int in [0, 31], or None for the one pixel).
        ``search_radius`` R (an int >= 0) bounds the window in level pixels and ``max_ratio`` (in (0, 1]) is the ratio
        test on SSD; see ``PointMatches``. Runs on every route, bank, ``out_dtype`` and ``peaks`` the records serve.
        The three arguments are checked before any GPU work (ValueError)."""
        radius, r, ratio = self._match_args(patch_radius, search_radius, max_ratio)
        levels, rows = self._record_rows(frames, points_capacity, None, radius)
        return self._records(*rows), self._matches(levels, rows, r, ratio)

    @staticmethod
    def _match_args(patch_radius, search_radius, max_ratio):
        return _ops.patch_radius(patch_radius), _ops.match_radius(search_radius), _ops.match_ratio(max_ratio)

    @staticmethod
    def _matches(levels, rows, search_radius, max_ratio):
        """``PointMatches`` of the rows ``_record_rows`` returns (every row found; its count is known on the host)."""
        points, values = rows[0], rows[3]
        count = torch.full((1,), points.shape[0], dtype=torch.int64, device=points.device)
        return PointMatches(*_ops.match_points(points, count, values, levels, search_radius, max_ratio))

    def run_host_matches(self, frames, patch_radius, search_radius, max_ratio=1.0, points_capacity=4096):
        """``run_frames_matches`` on host frames, as ``run_host_records`` takes them: numpy ``(PointRecords,
        PointMatches)``. The patches are matched on the device and never cross the host link: the records come without
        them, their values are the patch centres (the records of ``run_host_records`` without a patch, bit for bit).
        ``points_capacity`` sizes the first attempt; every point is returned. The arguments are checked before the
        upload."""
        radius, r, ratio = self._match_args(patch_radius, search_radius, max_ratio)
        staged, dev = self._stage_host(frames)

        def run(x):
            levels, rows = self._record_rows(x, points_capacity, None, radius)
            links = self._matches(levels, rows, r, ratio)
            values = rows[3] if radius is None else rows[3][:, radius, radius].contiguous()
            return rows[:3] + (values,) + tuple(links)
        outs = host_round_trip(staged, dev, run, lambda i, shape, dtype: torch.empty(shape, dtype=dtype, pin_memory=True))
        return self._records(*outs[:4]), PointMatches(*outs[4:])

    # -- frame-to-frame motion -------------------------------------------------------------------------------------------
    def run_frames_motion(self, frames, patch_radius, search_radius, max_ratio=1.0, threshold=MOTION_THRESHOLD,
                          hypotheses=MOTION_HYPOTHESES, seed=0, points_capacity=None):
        """``run_frames_matches`` and the motion between consecutive frames that its matches support
        (``PointRecords``, ``PointMatches``, ``PointMotion``), all CUDA tensors: per frame pair an affine map in frame
        pixels from a seeded RANSAC of ``hypotheses`` (an int in [1, 4096]) draws, inliers within ``threshold`` frame
        pixels (a real number > 0), refined by one least-squares step; see ``PointMotion``. ``seed`` (an int in
        [0, 2^64)) makes the draws reproducible. Runs on every route, bank, ``out_dtype``, ``frame_format`` and
        ``peaks`` the matches serve. Every argument is checked before any GPU work (ValueError)."""
        radius, r, ratio = self._match_args(patch_radius, search_radius, max_ratio)
        motion_args = _ops.motion_args(threshold, hypotheses, seed)
        levels, rows = self._record_rows(frames, points_capacity, None, radius)
        matches = self._matches(levels, rows, r, ratio)
        return self._records(*rows), matches, self._motion(rows, matches, *motion_args)

    @staticmethod
    def _motion(rows, matches, threshold, hypotheses, seed):
        """``PointMotion`` of the rows ``_record_rows`` returns and their ``PointMatches``."""
        points, frame_offsets, frame_yx = rows[:3]
        count = torch.full((1,), points.shape[0], dtype=torch.int64, device=points.device)
        return PointMotion(*_ops.estimate_motion(frame_offsets, frame_yx, matches.next, count, hypotheses, threshold,
                                                 seed))

    def run_host_motion(self, frames, patch_radius, search_radius, max_ratio=1.0, threshold=MOTION_THRESHOLD,
                        hypotheses=MOTION_HYPOTHESES, seed=0, points_capacity=4096):
        """``run_frames_motion`` on host frames, as ``run_host_matches`` takes them: numpy ``(PointRecords,
        PointMatches, PointMotion)``. The patches stay on the device: the records' values are the patch centres.
        ``points_capacity`` sizes the first attempt; every point is returned. The arguments are checked before the
        upload."""
        radius, r, ratio = self._match_args(patch_radius, search_radius, max_ratio)
        motion_args = _ops.motion_args(threshold, hypotheses, seed)
        staged, dev = self._stage_host(frames)

        def run(x):
            levels, rows = self._record_rows(x, points_capacity, None, radius)
            links = self._matches(levels, rows, r, ratio)
            motion = self._motion(rows, links, *motion_args)
            values = rows[3] if radius is None else rows[3][:, radius, radius].contiguous()
            return rows[:3] + (values,) + tuple(links) + tuple(motion)
        outs = host_round_trip(staged, dev, run, lambda i, shape, dtype: torch.empty(shape, dtype=dtype, pin_memory=True))
        return self._records(*outs[:4]), PointMatches(*outs[4:7]), PointMotion(*outs[7:])

    # -- host buffers on both sides (LineEndDisplayer.callback) -----------------------------------------------------------
    def run_host(self, frames, orient_out=None, line_end_out=None, points_capacity=4096):
        """frames: host numpy ``[B, H, W, 3]`` (``frame_format="nv12"``: ``[B, H * 3 / 2, W]`` uint8; ideally page-locked)
        -> host numpy results via the C-ABI host call (with ``orientations`` or ``peaks`` set, or off the ``PLAN``
        route: through ``run_frames`` and page-locked buffers, results ``[B * L, h, w, orientations]``). With
        ``out_dtype=torch.float16`` the results are ``np.float16``, and so must be ``orient_out`` / ``line_end_out``."""
        nb = self._bank_width() if self.orientations is not None else None
        if self._half():
            for name, arr in (("orient_out", orient_out), ("line_end_out", line_end_out)):
                if arr is not None and arr.dtype != np.float16:
                    raise ValueError("%s must be a np.float16 array for out_dtype=torch.float16, got %s" % (name, arr.dtype))
        frames = np.asarray(frames)
        nv12_hw = _ops.nv12_frame_hw(frames.shape, frames.dtype) if self._nv12() else None
        frames = np.ascontiguousarray(frames)
        if frames.ndim == (2 if nv12_hw else 3):
            frames = frames[np.newaxis]
        if frames.dtype != np.uint8:
            frames = frames.astype(np.float32)
        dev = self._device()
        tdtype = torch.uint8 if frames.dtype == np.uint8 else torch.float32
        # banks, peaks and the routes off PLAN go through run_frames (the C host-buffer call emits region maxima only)
        if nb is not None or self.peaks is not None or self._frame_route(nb, self.frame_format, tdtype,
                                                                          frames.shape) != PLAN:
            def run(x):   # through run_frames: the frames in and the results out through new page-locked buffers
                res = self.run_frames(x, points_capacity=points_capacity)
                return res.orient, res.padded_line_end, res.points
            orient, line_end, points = host_round_trip(torch.from_numpy(frames).pin_memory(), dev, run,
                                                       lambda i, shape, dtype: torch.empty(shape, dtype=dtype).pin_memory())
            if orient_out is not None:
                orient_out[...] = orient
                orient = orient_out
            if line_end_out is not None:
                line_end_out[...] = line_end
                line_end = line_end_out
            return LineEndResult(orient, line_end, None, points)
        if nv12_hw:
            plan = self._plan(nv12_hw + (3,), tdtype, dev, "nv12")
        else:
            plan = self._plan(frames.shape[1:], tdtype, dev)
        b = frames.shape[0]
        n = b * plan.levels
        out_np = np.float16 if self._half() else np.float32
        if orient_out is None:
            orient_out = np.empty((n, plan.h, plan.w, 3), out_np)
        if line_end_out is None:
            line_end_out = np.empty((n, plan.h, plan.w, 3), out_np)
        points = np.empty((points_capacity, 4), np.int64)
        count = ctypes.c_int64(0)
        name = "silent_pipeline_run_host_f16" if self._half() else "silent_pipeline_run_host"
        with torch.cuda.device(dev):
            _lib.check(getattr(_lib.lib(), name)(
                plan.handle, ctypes.byref(self.stack_weights()), frames.ctypes.data, b, orient_out.ctypes.data,
                line_end_out.ctypes.data, points.ctypes.data, points_capacity, ctypes.byref(count),
                _ops.stream_ptr()), name)
        if count.value > points_capacity:
            # rare (an all-zero level emits every pixel, top_value_points.py:42-44): redo with room for every point, as
            # run_frames does -- feature points are never silently truncated
            return self.run_host(frames, orient_out, line_end_out, points_capacity=int(count.value))
        return LineEndResult(orient_out, line_end_out, None, points[:count.value])

    def callback(self, frame, cam_id=None, depth=2):
        """Per-frame entry point with the reference's signature (``recognition_testing.py:136-144``).

        Returns ``[frame, [orient level images...], [padded_line_end level images...], points]``: the two result
        tensors on the north-star path as per-level host images, plus the feature points the reference builds but never
        fetches. ``frame`` is the frame as given (an NV12 array with ``frame_format="nv12"``).
        """
        res = self.run_host(np.asarray(frame))
        return [frame, [res.orient[i] for i in range(res.orient.shape[0])],
                [res.padded_line_end[i] for i in range(res.padded_line_end.shape[0])], res.points]
