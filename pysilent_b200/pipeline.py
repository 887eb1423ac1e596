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
from .util.zoom.from_image import PyramidPlan

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


LineEndResult = collections.namedtuple("LineEndResult", "orient padded_line_end gray points")
LineEndResult.__doc__ = """orient: ``orient_tensor`` [N,h,w,3]; padded_line_end: ``padded_line_end_tensor`` [N,h,w,3];
gray: ``gray_line_end_tensor`` [N,h,w,1] (or None); points: int64 [K,4] rows (level, y, x, 0) (``top_percent_points``)."""


class LineEndPipeline:
    """Drop-in for the compute half of ``LineEndDisplayer`` (camera / window handling is out of scope).

    Constructor keywords follow ``PyramidDisplayer.__init__`` (``pyramid_displayer.py:22``): ``output_size`` is
    ``(w, h)`` of every pyramid level, ``zoom_ratio`` the scale between levels.
    """

    def __init__(self, n_dimensions=2, output_size=(288, 192), output_colors=3, zoom_ratio=math.e ** .5, device=None,
                 orientations=None):
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

    def _region(self):
        rh, rw = self.region_shape[1], self.region_shape[2]
        if int(rh) != rh or int(rw) != rw:
            raise ValueError("Ambiguous dimension: %s" % ([rh, rw],))
        return int(rh), int(rw)

    # -- graph on a pyramid (LineEndDisplayer.run) --------------------------------------------------------------------
    def run(self, pyramid_tensor, want_points=True):
        """S1-S8 on a pyramid ``[N, h, w, 3]`` (numpy or CUDA tensor). One fused kernel + the emit kernels."""
        if self.orientations is not None:
            return self.run_bank(pyramid_tensor, want_points)
        if self.blur_size != 7:
            return self.run_unfused(pyramid_tensor, want_points)
        x = _ops.as_device_tensor(pyramid_tensor)
        # the fused kernels skip exact-zero weights and shortcut the regulator where the blur is provably >= 1: valid for
        # finite input only (include/silent_b200.h). NaN / Inf / huge values go operator by operator, like the graph.
        if not bool((x.abs() <= _ops.FUSED_INPUT_MAX).all()):
            return self.run_unfused(x, want_points)
        orient, line_end, gray = _ops.stack_fused(x, self.stack_weights())
        points = None
        if want_points:
            rh, rw = self._region()
            points = _ops.max_value_indices_region(gray, rh, rw)
        return LineEndResult(orient, line_end, gray, points)

    def run_unfused(self, pyramid_tensor, want_points=True):
        """The same graph through the per-operator kernels (any filter structure, any blur size)."""
        from .filters import rgc_filter, rgby_filter, orientation_filter
        from .util.selection import pad_inwards, max_value_indices_region
        from .util.color import get_value_from_color
        x = _ops.as_device_tensor(pyramid_tensor)
        orient = orientation_filter(rgby_filter(rgc_filter(x)), self.blur_size)
        line_end = _ops.conv2d(orient, self.simplex_end_stop, post=_lib.POST_RELU_CLIP, clip_max=255.0)
        padded = pad_inwards(line_end, [[0, 0], [2, 2], [2, 2], [0, 0]])
        gray = get_value_from_color(padded)
        points = max_value_indices_region(padded, self.region_shape, gray) if want_points else None
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

    def run_bank(self, pyramid_tensor, want_points=True):
        """Config C4: S1-S2 on 3 channels, S3-S7 on an ``orientations``-channel bank (same composition as ``compile()``,
        ``recognition_testing.py:69-77``). Up to 8 orientations through the per-operator kernels; 12 and 16 through the
        fused bank stack (``silent_stack_bank``), which needs a finite pyramid."""
        from .util.selection import pad_inwards, max_value_indices_region
        from .util.color import get_value_from_color
        from .util.regulator import regulate_tensor
        nb = self._bank_width()
        x = _ops.as_device_tensor(pyramid_tensor)
        region = [1, self.region_shape[1], self.region_shape[2], nb]
        if nb > 8:
            if not bool((x.abs() <= _ops.FUSED_INPUT_MAX).all()):
                raise ValueError("a pyramid with NaN, Inf or values beyond 1e30 goes operator by operator, which supports "
                                 "at most 8 orientations (got %d)" % nb)
            orient, padded, gray = _ops.stack_bank(x, self.orientation_bank())
            points = max_value_indices_region(padded, region, gray) if want_points else None
            return LineEndResult(orient, padded, gray, points)
        f = self.bank_filters()
        x = _ops.conv2d(_ops.conv2d(x, f["rgc"], post=_lib.POST_RELU), f["rgby"], post=_lib.POST_RELU)
        orient = regulate_tensor(_ops.conv2d(x, f["stripe"], post=_lib.POST_RELU), f["blur"], 1.0, .1)
        line_end = _ops.conv2d(orient, f["end"], post=_lib.POST_RELU_CLIP, clip_max=255.0)
        padded = pad_inwards(line_end, [[0, 0], [2, 2], [2, 2], [0, 0]])
        gray = get_value_from_color(padded)
        points = max_value_indices_region(padded, region, gray) if want_points else None
        return LineEndResult(orient, padded, gray, points)

    # -- frames resident in HBM ---------------------------------------------------------------------------------------
    def _plan(self, frame_shape, frame_dtype, device):
        """Plan cache keyed like the reference's per-shape session (``recognition_testing.py:108-118``). The cache is
        per pipeline: use one ``LineEndPipeline`` per camera thread, as the reference uses one displayer per camera."""
        key = (tuple(int(v) for v in frame_shape), frame_dtype, self.output_colors, self.output_size,
               float(self.zoom_ratio), str(device))
        plan = self._plans.get(key)
        if plan is None:
            with torch.cuda.device(device):
                plan = PyramidPlan(frame_shape, frame_dtype, self.output_colors, self.output_size, self.zoom_ratio)
            self._plans[key] = plan
        return plan

    def plan_for(self, frames):
        return self._plan(frames.shape[1:], frames.dtype, frames.device)

    def run_frames(self, frames, want_points=True, points_capacity=None, out=None):
        """frames: CUDA ``[B, H, W, 3]`` uint8/float32 -> LineEndResult over ``B * L`` levels (pyramid + S1-S8).

        ``out`` may carry preallocated ``(orient, padded_line_end, points, count)`` tensors to avoid allocation in a
        steady-state loop; ``points`` then holds ``count`` valid rows (no host sync is performed in that case).
        """
        nb = self._bank_width() if self.orientations is not None else None
        frames = frames if frames.dim() == 4 else frames.unsqueeze(0)
        frames = frames.contiguous()
        if nb is not None:   # config C4 and its variants
            if nb in _lib.FUSED_BANK_WIDTHS and frames.dtype == torch.uint8 and frames.shape[3] >= 3 \
                    and self.blur_size == 7 and self.output_colors == 3 and (frames.shape[2] * frames.shape[3]) % 16 == 0:
                return self._run_frames_bank(frames, want_points, points_capacity)   # fused: 4 kernels + emit
            from .util.zoom.from_image import image_to_zoom_tensor   # other frames: pyramid, then run_bank
            return self.run_bank(image_to_zoom_tensor(frames, self.output_colors, self.output_size, self.zoom_ratio),
                                 want_points)
        plan = self.plan_for(frames)
        b = int(frames.shape[0])
        plan.reserve(b)
        n = b * plan.levels
        dev = frames.device
        if out is None:
            orient = torch.empty((n, plan.h, plan.w, 3), dtype=torch.float32, device=dev)
            line_end = torch.empty_like(orient)
            cap = int(points_capacity) if points_capacity else max(64 * n, 1024)
            points = torch.empty((cap, 4), dtype=torch.int64, device=dev)
            count = torch.zeros(1, dtype=torch.int64, device=dev)
        else:
            orient, line_end, points, count = out
            cap = int(points.shape[0])
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().silent_pipeline_run(
                plan.handle, ctypes.byref(self.stack_weights()), _ops.ptr(frames), b, None, _ops.ptr(orient),
                _ops.ptr(line_end), _ops.ptr(points), cap, _ops.ptr(count) if want_points else None,
                _ops.stream_ptr()), "silent_pipeline_run")
        if out is not None:
            return LineEndResult(orient, line_end, None, points)
        if not want_points:
            return LineEndResult(orient, line_end, None, None)
        total = int(count.item())
        if total > cap:   # rare (e.g. an all-black level emits every pixel): redo the emit with room for everything
            return self.run_frames(frames, want_points, points_capacity=total)
        return LineEndResult(orient, line_end, None, points[:total])

    def _run_frames_bank(self, frames, want_points=True, points_capacity=None):
        """Config C4 fused: pyramid_pair_kernel -> stack_a (rgc, rgby) -> stack_bank_kernel (stripe bank, regulator,
        depthwise end bank, mask, mean) -> emit, through ``silent_pipeline_run_orientations``."""
        plan = self.plan_for(frames)
        b = int(frames.shape[0])
        plan.reserve(b)
        n, dev = b * plan.levels, frames.device
        bank = self.orientation_bank()
        orient = torch.empty((n, plan.h, plan.w, bank.orientations), dtype=torch.float32, device=dev)
        line_end = torch.empty_like(orient)
        cap = int(points_capacity) if points_capacity else max(64 * n, 1024)
        points = torch.empty((cap, 4), dtype=torch.int64, device=dev)
        count = torch.zeros(1, dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().silent_pipeline_run_orientations(
                plan.handle, ctypes.byref(bank), _ops.ptr(frames), b, _ops.ptr(orient), _ops.ptr(line_end),
                _ops.ptr(points), cap, _ops.ptr(count) if want_points else None, _ops.stream_ptr()),
                "silent_pipeline_run_orientations")
        if not want_points:
            return LineEndResult(orient, line_end, None, None)
        total = int(count.item())
        if total > cap:
            return self._run_frames_bank(frames, want_points, points_capacity=total)
        return LineEndResult(orient, line_end, None, points[:total])

    # -- host buffers on both sides (LineEndDisplayer.callback) -----------------------------------------------------------
    def run_host(self, frames, orient_out=None, line_end_out=None, points_capacity=4096):
        """frames: host numpy ``[B, H, W, 3]`` (ideally page-locked) -> host numpy results via the C-ABI host call (with
        ``orientations`` set: through ``run_frames`` and page-locked buffers, results ``[B * L, h, w, orientations]``)."""
        if self.orientations is not None:
            self._bank_width()
        frames = np.ascontiguousarray(frames)
        if frames.ndim == 3:
            frames = frames[np.newaxis]
        if frames.dtype != np.uint8:
            frames = frames.astype(np.float32)
        dev = self._device()
        if self.orientations is not None:
            return self._run_host_bank(frames, dev, orient_out, line_end_out, points_capacity)
        tdtype = torch.uint8 if frames.dtype == np.uint8 else torch.float32
        plan = self._plan(frames.shape[1:], tdtype, dev)
        b = frames.shape[0]
        n = b * plan.levels
        if orient_out is None:
            orient_out = np.empty((n, plan.h, plan.w, 3), np.float32)
        if line_end_out is None:
            line_end_out = np.empty((n, plan.h, plan.w, 3), np.float32)
        points = np.empty((points_capacity, 4), np.int64)
        count = ctypes.c_int64(0)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().silent_pipeline_run_host(
                plan.handle, ctypes.byref(self.stack_weights()), frames.ctypes.data, b, orient_out.ctypes.data,
                line_end_out.ctypes.data, points.ctypes.data, points_capacity, ctypes.byref(count),
                _ops.stream_ptr()), "silent_pipeline_run_host")
        if count.value > points_capacity:
            # rare (an all-zero level emits every pixel, top_value_points.py:42-44): redo with room for every point, as
            # run_frames does -- feature points are never silently truncated
            return self.run_host(frames, orient_out, line_end_out, points_capacity=int(count.value))
        return LineEndResult(orient_out, line_end_out, None, points[:count.value])

    def _run_host_bank(self, frames, dev, orient_out, line_end_out, points_capacity):
        """run_host for a bank: the frames go up from a page-locked copy, and the results come back with asynchronous
        copies into page-locked buffers and one synchronisation, as ``LineEndDisplayer.callback`` does."""
        staged = torch.from_numpy(frames).pin_memory()
        with torch.cuda.device(dev):
            res = self.run_frames(staged.to(dev, non_blocking=True), points_capacity=points_capacity)
            host = []
            for t in (res.orient, res.padded_line_end, res.points):
                h = torch.empty(tuple(t.shape), dtype=t.dtype).pin_memory()
                h.copy_(t, non_blocking=True)
                host.append(h)
            torch.cuda.current_stream().synchronize()
        orient, line_end, points = (h.numpy() for h in host)
        if orient_out is not None:
            orient_out[...] = orient
            orient = orient_out
        if line_end_out is not None:
            line_end_out[...] = line_end
            line_end = line_end_out
        return LineEndResult(orient, line_end, None, points)

    def callback(self, frame, cam_id=None, depth=2):
        """Per-frame entry point with the reference's signature (``recognition_testing.py:136-144``).

        Returns ``[frame, [orient level images...], [padded_line_end level images...], points]``: the two result
        tensors on the north-star path as per-level host images, plus the feature points the reference builds but never
        fetches.
        """
        res = self.run_host(np.asarray(frame))
        return [frame, [res.orient[i] for i in range(res.orient.shape[0])],
                [res.padded_line_end[i] for i in range(res.padded_line_end.shape[0])], res.points]
