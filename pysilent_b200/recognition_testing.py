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
from .pipeline import LineEndPipeline
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
            rh, rw = region_dims(self.centroid_region_shape)
            state_shape = (shape[0], -(-shape[1] // rh), -(-shape[2] // rw), 1)
            if self.pyramid_tensor_shape != shape or self.energy_values is None:                  # pre_compile, :45-57
                self.pyramid_tensor_shape = shape
                self.energy_values = torch.full(state_shape, 8.0, dtype=torch.float32, device=gray.device)
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

    def run(self, pyramid_tensor):
        """``pyramid_tensor`` ``[L, h, w, 3]`` -> the six fetched tensors as host arrays (``session.run``, ``:132``)."""
        res = LineEndPipeline.run(self, pyramid_tensor, want_points=False)
        return [t.cpu().numpy() for t in self.display_tensors(res.orient, res.padded_line_end, res.gray)]

    def run_frames_display(self, frames):
        """Frames resident in HBM ``[B, H, W, 3]`` -> the six display tensors on the device (``B * L`` levels). With
        ``B`` > 1 every frame is an independent camera stream with its own slice of the boosting state."""
        res = self.run_frames(frames, want_points=False)
        return self.display_tensors(res.orient, res.padded_line_end)

    def callback(self, frame, cam_id=None, depth=2):
        """``recognition_testing.py:136-144``: ``[frame] + [[tensors[x][y] for y in levels] for x in range(6)]``."""
        if self.orientations is not None:
            self._bank_width()
        z = np.asarray(frame)
        z = np.ascontiguousarray(z if z.dtype == np.uint8 else z.astype(np.float32))
        dev = self._device()
        self._slot = (self._slot + 1) % self.host_slots
        # frame in through a page-locked buffer (asynchronous H2D), the six tensors out into page-locked buffers with
        # asynchronous copies and ONE synchronisation -- instead of a pageable upload and six blocking .cpu() calls
        staged = self._host_buffer(("frame", self._slot), z.shape, torch.uint8 if z.dtype == np.uint8 else torch.float32)
        staged.numpy()[...] = z
        with torch.cuda.device(dev):
            tensors = self.run_frames_display(staged.to(dev, non_blocking=True).unsqueeze(0))
            outs = []
            for i, t in enumerate(tensors):
                host = self._host_buffer(("out", self._slot, i), tuple(t.shape), t.dtype)
                host.copy_(t, non_blocking=True)
                outs.append(host.numpy())
            torch.cuda.current_stream().synchronize()
        return [frame] + [[outs[x][y] for y in range(len(outs[x]))] for x in range(6)]

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
