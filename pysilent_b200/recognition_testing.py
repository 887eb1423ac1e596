"""``LineEndDisplayer``: the reference's per-frame driver class on the B200 kernels.

Reference: ``slam_recognition/recognition_testing.py:18-144``. ``callback(frame, cam_id)`` builds the foveated pyramid,
runs the filter stack and returns ``[frame] + six lists of per-level images`` -- ``orient_tensor``,
``255 - centroids * 255``, ``255 - centroids2 * 255``, ``fired_importants * 255``, ``update_importances`` and
``padded_line_end_tensor`` (``:98-100, 132, 144``). The boosting state (``energy_values``, a ``tf.Variable`` there) is a
CUDA tensor owned by the displayer; it is re-initialised to 8 whenever the pyramid shape changes, as the reference
re-creates its graph and variables (``:108-118``). Camera capture and windows (``PyramidDisplayer.run_camera``) are out
of scope: feed frames to ``callback`` / ``display`` directly.
"""
import math as m

import numpy as np
import torch

from . import _lib, _ops
from .pipeline import LineEndPipeline, host_round_trip
from .util.centroids import get_centroids, _region as region_dims
from .util.color import get_value_from_color
from .util.energy.boosting import get_boosting, initialize_boosting
from .util.energy.recovery import recovery_mode

debug = True


class LineEndDisplayer(LineEndPipeline):
    def __init__(self, n_dimensions=2, **argv):
        """Line-end ("end-stopped") detector stage on top of the pyramid pipeline; same constructor attributes as the
        reference's ``LineEndDisplayer.__init__`` (``recognition_testing.py:22-43``)."""
        super(LineEndDisplayer, self).__init__(n_dimensions, **argv)
        if self.out_dtype != torch.float32:   # the display chain reads float32 padded_line_end
            raise ValueError("LineEndDisplayer computes its display images from float32 outputs; out_dtype must be "
                             "torch.float32, got %s" % (self.out_dtype,))
        self.tensor_return_type = [torch.Tensor]
        self.precompile_list = []
        self.constant_recovery = True
        self.input_based_recovery = False
        self.excitation_max = 8
        self.top_percent_pool = .5
        self.rotation_invariance = False
        self.padded_firing = None
        self.centroid_region_shape = [1, 3, 3]  # block size of the centroid / importance pooling (reference default)
        self.pyramid_tensor_shape = None
        self.energy_values = None
        # page-locked host buffers of callback(): a ring of `host_slots` sets, so the arrays handed out by one call stay
        # untouched for the next host_slots - 1 calls (the reference returns fresh arrays; a consumer that keeps frames
        # longer copies them)
        self.host_slots = 3
        self._slot = -1
        self._pinned = {}

    # -- the part of compile() after gray_line_end_tensor (recognition_testing.py:79-100) -------------------------------
    def display_tensors(self, orient, padded_line_end, gray=None, fused=True):
        """Device tensors in the order ``run()`` fetches them; updates ``energy_values``. ``fused`` (default) runs the
        chain as the two launches of ``silent_display_tensors``; ``fused=False`` composes the stand-alone operators one by
        one, as the reference graph is written (same bits, seventeen launches)."""
        if gray is None:
            gray = get_value_from_color(padded_line_end)                                          # :77
        shape = tuple(orient.shape)
        half = (np.asarray(shape[1:3], dtype=np.float32) / np.float32(m.e ** .5)).astype(np.int32)   # :82
        if fused:
            rh, rw = self._boosting_state(shape, gray.device)
            cent, cent2, fired, update = _ops.display_tensors(gray, self.energy_values, rh, rw, int(half[0]), int(half[1]),
                                                              1, 1, recovery_mode(False, True))   # :79-87
            return [orient, cent, cent2, fired, update, padded_line_end]                          # :98-100
        centroids, importances = get_centroids(_ops.pointwise(gray, _lib.PW_DIV255), self.centroid_region_shape,
                                               debug=True)                                        # :79-80
        importances = _ops.pointwise(importances, _lib.PW_IMPORTANCE)                             # :81
        im2 = _ops.resize_nearest(gray, int(half[0]), int(half[1]))                               # :83
        centroids2, _ = get_centroids(_ops.pointwise(im2, _lib.PW_DIV255), self.centroid_region_shape, debug=True)
        if self.pyramid_tensor_shape != shape or self.energy_values is None:                      # pre_compile, :45-57
            self.pyramid_tensor_shape = shape
            self.energy_values = initialize_boosting(importances)
        fired_importants, update_importances = get_boosting(importances, self.energy_values,
                                                            for_visualizing=True)                 # :86-87
        return [orient, _ops.pointwise(centroids, _lib.PW_INVERT255), _ops.pointwise(centroids2, _lib.PW_INVERT255),
                _ops.pointwise(fired_importants, _lib.PW_MUL255), update_importances, padded_line_end]   # :98-100

    def _boosting_state(self, shape, device):
        """Re-initialise ``energy_values`` to 8 when the per-step shape ``(levels, h, w, C)`` changes (pre_compile,
        ``:45-57``); returns the centroid region ``(rh, rw)``."""
        rh, rw = region_dims(self.centroid_region_shape)
        if self.pyramid_tensor_shape != shape or self.energy_values is None:
            self.pyramid_tensor_shape = shape
            self.energy_values = torch.full((shape[0], -(-shape[1] // rh), -(-shape[2] // rw), 1), 8.0,
                                            dtype=torch.float32, device=device)
        return rh, rw

    def run(self, pyramid_tensor):
        """``pyramid_tensor`` ``[L, h, w, 3]`` -> the six fetched tensors as host arrays (``session.run``, ``:132``)."""
        res = LineEndPipeline.run(self, pyramid_tensor, want_points=False)
        return [t.cpu().numpy() for t in self.display_tensors(res.orient, res.padded_line_end, res.gray)]

    def run_frames_display(self, frames):
        """Frames resident in HBM ``[B, H, W, 3]`` -> the six display tensors on the device (``B * L`` levels). With
        ``B`` > 1 every frame is an independent camera stream with its own slice of the boosting state."""
        res = self.run_frames(frames, want_points=False)
        return self.display_tensors(res.orient, res.padded_line_end)

    def run_clip(self, frames):
        """A clip of consecutive frames resident in HBM -> the six display tensors on the device, in the order of
        ``run_frames_display``. ``frames`` is ``[T, H, W, 3]`` (one camera) or ``[T, S, H, W, 3]`` (S cameras),
        time-major (``frame_format="nv12"``: ``[T, H * 3 / 2, W]`` or ``[T, S, H * 3 / 2, W]``); step t's images are ``[t * S * L, (t + 1) * S * L)`` and equal, bit for bit, what
        ``run_frames_display(frames[t])`` returns when called for t = 0 ... T-1 in turn. ``energy_values`` ends where
        those calls leave it, so ``callback``, ``run_clip`` and ``callback`` on one camera continue one state. The
        pipeline runs once over all T * S frames, and the boosting recurrence over the whole clip in one launch."""
        rank = frames.dim() if isinstance(frames, torch.Tensor) else np.ndim(frames)
        frame_rank = 2 if self._nv12() else 3
        if self._nv12():
            _ops.nv12_frame_hw(frames.shape, frames.dtype, ranks=(3, 4), what="NV12 clips")
        if rank not in (frame_rank + 1, frame_rank + 2) or frames.shape[0] < 1:
            raise ValueError("run_clip takes frames [T, H, W, 3] or [T, S, H, W, 3] with T >= 1, got shape %s"
                             % (tuple(frames.shape),))
        steps = int(frames.shape[0])
        res = self.run_frames(frames.reshape((-1,) + tuple(frames.shape[-frame_rank:])), want_points=False)
        orient, padded = res.orient, res.padded_line_end
        gray = get_value_from_color(padded)                                                       # :77
        step_shape = (orient.shape[0] // steps,) + tuple(orient.shape[1:])
        half = (np.asarray(step_shape[1:3], dtype=np.float32) / np.float32(m.e ** .5)).astype(np.int32)   # :82
        rh, rw = self._boosting_state(step_shape, gray.device)
        cent, cent2, fired, update = _ops.display_sequence(gray, self.energy_values, steps, rh, rw, int(half[0]),
                                                           int(half[1]), 1, 1, recovery_mode(False, True))
        return [orient, cent, cent2, fired, update, padded]

    def callback_clip(self, frames, cam_id=None):
        """``callback`` over a host clip ``[T, H, W, 3]`` (``frame_format="nv12"``: ``[T, H * 3 / 2, W]``) of one
        camera: a list of T results, each
        ``[frames[t]] + six lists of per-level images`` like ``callback``'s, with the state carried from step to step.
        The clip goes up through a page-locked buffer, runs through ``run_clip`` and comes back with asynchronous
        copies and one synchronisation. The arrays handed out stay untouched for the next ``host_slots - 1`` calls of
        ``callback`` or ``callback_clip``."""
        z = np.asarray(frames)
        if self._nv12():
            _ops.nv12_frame_hw(z.shape, z.dtype, ranks=(3,), what="NV12 clips")
        elif z.ndim != 4 or z.shape[0] < 1:
            raise ValueError("callback_clip takes host frames [T, H, W, 3] with T >= 1, got shape %s" % (z.shape,))
        if self.orientations is not None:
            self._bank_width()
        outs = self._round_trip("clip", z, self.run_clip)
        L = outs[0].shape[0] // z.shape[0]
        return [[frames[t]] + [[outs[x][t * L + y] for y in range(L)] for x in range(6)] for t in range(z.shape[0])]

    def callback(self, frame, cam_id=None, depth=2):
        """``recognition_testing.py:136-144``: ``[frame] + [[tensors[x][y] for y in levels] for x in range(6)]``. With
        ``frame_format="nv12"`` the frame is one NV12 array ``[H * 3 / 2, W]``, and comes back as given."""
        if self.orientations is not None:
            self._bank_width()
        z = np.asarray(frame)
        if self._nv12():
            _ops.nv12_frame_hw(z.shape, z.dtype, ranks=(2,))
        outs = self._round_trip("frame", z, lambda x: self.run_frames_display(x.unsqueeze(0)))
        return [frame] + [[outs[x][y] for y in range(len(outs[x]))] for x in range(6)]

    def _round_trip(self, kind, z, run):
        """``host_round_trip`` of the frames ``z`` through the next slot of the page-locked buffer ring: one
        synchronisation instead of a pageable upload and six blocking ``.cpu()`` calls."""
        z = np.ascontiguousarray(z if z.dtype == np.uint8 else z.astype(np.float32))
        dev = self._device()
        self._slot = slot = (self._slot + 1) % self.host_slots
        staged = self._host_buffer((kind, slot), z.shape, torch.uint8 if z.dtype == np.uint8 else torch.float32)
        staged.numpy()[...] = z
        return host_round_trip(staged, dev, run, lambda i, shape, dtype: self._host_buffer((kind, slot, i), shape, dtype))

    def _host_buffer(self, key, shape, dtype):
        buf = self._pinned.get(key)
        if buf is None or tuple(buf.shape) != tuple(shape) or buf.dtype != dtype:
            buf = torch.empty(tuple(shape), dtype=dtype).pin_memory()
            self._pinned[key] = buf
        return buf

    def display(self, frame, cam_id=None):
        """``PyramidDisplayer.display`` (``pyramid_displayer.py:35-40``): everything scaled by 1/255 for the windows."""
        frame_from_callback = self.callback(frame, cam_id)
        return [np.array(frame_from_callback[x]) / 255.0 for x in range(len(frame_from_callback))]
