"""Foveated pyramid build on the GPU. Reference: ``slam_recognition/util/zoom/from_image.py:10-69``."""
import ctypes
import threading

import numpy as np
import torch

from ... import _lib, _ops


class PyramidPlan:
    """Owns a ``silent_plan`` (level geometry + order-5 spline tap tables, uploaded once). ``frame_shape`` is
    ``(H, W, C)``; with ``frame_format="nv12"`` the frames are NV12 ``[H * 3 / 2, W]`` uint8 arrays of an H x W x 3
    image (``C`` = 3), converted on the GPU before the pyramid reads them."""

    def __init__(self, frame_shape, frame_dtype, num_colors, center_dimensions, scale, frame_format="bgr"):
        h, w, c = (int(v) for v in frame_shape)
        if frame_format == "nv12":
            dtype = _lib.SILENT_NV12
        else:
            dtype = _lib.SILENT_U8 if frame_dtype == torch.uint8 else _lib.SILENT_F32
        self.params = _lib.SilentParams(h, w, c, int(num_colors), int(center_dimensions[0]), int(center_dimensions[1]),
                                        float(scale), dtype, 0)
        self.handle = ctypes.c_void_p()
        _lib.check(_lib.lib().silent_plan_create(ctypes.byref(self.params), ctypes.byref(self.handle)),
                   "silent_plan_create")
        self.levels = _lib.lib().silent_plan_levels(self.handle)
        self.h, self.w = int(center_dimensions[1]), int(center_dimensions[0])
        self.num_colors = int(num_colors)
        self.frame_dtype = frame_dtype
        self.frame_format = frame_format

    def level_info(self, level):
        vals = [ctypes.c_int() for _ in range(6)]
        _lib.check(_lib.lib().silent_plan_level_info(self.handle, level, *[ctypes.byref(v) for v in vals]))
        return tuple(v.value for v in vals)

    def level_tables(self, level):
        iy = np.empty((self.h, 6), np.int32)
        wy = np.empty((self.h, 6), np.float32)
        ix = np.empty((self.w, 6), np.int32)
        wx = np.empty((self.w, 6), np.float32)
        _lib.check(_lib.lib().silent_plan_level_tables(self.handle, level, iy.ctypes.data, wy.ctypes.data,
                                                       ix.ctypes.data, wx.ctypes.data))
        return iy, wy, ix, wx

    def level_coords(self, level):
        """``(frame_y [h], frame_x [w])`` float32: the frame position of every row and column of ``level``, NaN where
        the level defines the row or column as 0 (``silent_plan_level_coords``)."""
        fy = np.empty(self.h, np.float32)
        fx = np.empty(self.w, np.float32)
        _lib.check(_lib.lib().silent_plan_level_coords(self.handle, level, fy.ctypes.data, fx.ctypes.data))
        return fy, fx

    @property
    def algorithmic_bytes(self):
        return int(_lib.lib().silent_plan_algorithmic_bytes(self.handle))

    def reserve(self, batch):
        _lib.check(_lib.lib().silent_plan_reserve(self.handle, int(batch)), "silent_plan_reserve")

    def build(self, frames):
        """``frames`` CUDA ``[B, H, W, C]`` of the plan's dtype (NV12 plans: ``[B, H * 3 / 2, W]`` uint8) ->
        ``[B * L, h, w, num_colors]`` float32."""
        b = int(frames.shape[0])
        out = torch.empty((b * self.levels, self.h, self.w, self.num_colors), dtype=torch.float32, device=frames.device)
        if self.levels > 0:
            if self.frame_format == "nv12":
                self.reserve(b)   # the converted frames live in the plan's workspace
            with torch.cuda.device(frames.device):
                _lib.check(_lib.lib().silent_pyramid_build(self.handle, _ops.ptr(frames), b, _ops.ptr(out),
                                                           _ops.stream_ptr()), "silent_pyramid_build")
        return out

    def __del__(self):
        try:
            if self.handle:
                _lib.lib().silent_plan_destroy(self.handle)
                self.handle = ctypes.c_void_p()
        except Exception:
            pass


_plans = {}
_plans_lock = threading.Lock()


def get_plan(frame_shape, frame_dtype, num_colors, center_dimensions, scale, device):
    """Plan cache keyed by everything the geometry depends on (the reference rebuilds its graph on shape change,
    ``recognition_testing.py:108-118``)."""
    key = (tuple(int(v) for v in frame_shape), frame_dtype, int(num_colors), tuple(int(v) for v in center_dimensions),
           float(scale), str(device))
    with _plans_lock:
        plan = _plans.get(key)
        if plan is None:
            with torch.cuda.device(device):
                plan = PyramidPlan(frame_shape, frame_dtype, num_colors, center_dimensions, scale)
            _plans[key] = plan
    return plan


def image_to_zoom_tensor(image, num_colors, center_dimensions, scale):
    """Convert an image (or a batch of images) to its foveated pyramid.

    Each level takes a ``scale``-times larger centred crop of the image and resamples it to ``center_dimensions`` with
    the order-5 spline of ``scipy.ndimage.zoom(prefilter=False)``; results match the reference to float32 rounding.

    :param image: ``[H, W, C]`` or ``[B, H, W, C]``; numpy or torch; uint8 or float (values are NOT rescaled).
    :param num_colors: channels ``0..num_colors-1`` are used.
    :param center_dimensions: ``(w, h)`` of every level (reversed internally, like the reference).
    :param scale: ratio between the crops of consecutive levels, > 1.
    :return: CUDA float32 ``[L, h, w, num_colors]`` (``[B * L, ...]`` for a batch). Rows/columns the reference leaves
        uninitialised (``np.empty``) are 0.
    """
    frames, plan = zoom_frames_and_plan(image, num_colors, center_dimensions, scale)
    return plan.build(frames)


def zoom_frames_and_plan(image, num_colors, center_dimensions, scale):
    """The batch ``[B, H, W, C]`` (CUDA, uint8 or float32) that ``image_to_zoom_tensor`` builds its pyramid from, and
    the cached ``PyramidPlan`` it builds it with (whose geometry places each level's pixels in the frame)."""
    assert scale > 1, "Scale must be greater than one."
    assert num_colors > 0, "Number of colors must be greater than zero."
    for d in center_dimensions:
        assert d > 0, "Each dimension must be larger than zero."
    if isinstance(image, np.ndarray):
        image = torch.from_numpy(np.ascontiguousarray(image if image.dtype == np.uint8 else image.astype(np.float32)))
    if not isinstance(image, torch.Tensor):
        raise TypeError("image must be a numpy array or torch tensor")
    if image.dtype != torch.uint8:
        image = image.to(torch.float32)
    _ops._require_cuda()
    image = image.cuda() if not image.is_cuda else image
    batched = image.dim() == 4
    frames = (image if batched else image.unsqueeze(0)).contiguous()
    if frames.dim() != 4:
        raise ValueError("image must be [H, W, C] or [B, H, W, C], got shape %s" % (tuple(image.shape),))
    plan = get_plan(frames.shape[1:], frames.dtype, num_colors, center_dimensions, scale, frames.device)
    if plan.levels < 0:
        raise ValueError("negative dimensions are not allowed")
    return frames, plan
