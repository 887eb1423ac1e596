"""Device-side operator implementations over the C ABI. torch supplies device memory and streams only.

Tensors are contiguous float32 NHWC ``[levels, h, w, C]`` on a CUDA device (the reference's placeholder layout,
``recognition_testing.py:62``); numpy inputs are uploaded to the current CUDA device.
"""
import ctypes
import math
import numbers
import threading

import numpy as np
import torch

from . import _lib

_weights_lock = threading.Lock()
_weights_cache = {}


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("pysilent_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.")


# largest input magnitude the fused stack accepts: no stage can overflow to Inf from here (the five filters together
# amplify by well under 1e6), so every intermediate of the fused kernels stays finite until the regulator's own 0 * inf
FUSED_INPUT_MAX = 1.0e30


def fused_input_ok(x):
    """Whether the fused stacks may take the tensor ``x``: no NaN, no Inf and no magnitude beyond FUSED_INPUT_MAX."""
    return bool((x.abs() <= FUSED_INPUT_MAX).all())


def as_device_tensor(t, dtype=torch.float32):
    """torch CUDA / numpy -> contiguous CUDA tensor of ``dtype``."""
    _require_cuda()
    if isinstance(t, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(t)).cuda()
    elif not isinstance(t, torch.Tensor):
        raise TypeError("expected a torch.Tensor or numpy array, got %r" % type(t))
    if not t.is_cuda:
        t = t.cuda()
    if t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def filter_on_device(filt, device):
    """HWIO filter (numpy float64 from the generators, or a tensor) -> float32 CUDA tensor; cached by content."""
    if isinstance(filt, torch.Tensor):
        return filt.to(device=device, dtype=torch.float32).contiguous()
    a = np.ascontiguousarray(np.asarray(filt), dtype=np.float32)   # tf.constant(..., dtype=tf.float32) rounding
    key = (a.shape, a.tobytes(), str(device))
    with _weights_lock:
        t = _weights_cache.get(key)
        if t is None:
            if len(_weights_cache) > 256:
                _weights_cache.clear()
            t = torch.from_numpy(a).to(device)
            _weights_cache[key] = t
    return t


def _nhwc(t, what):
    if t.dim() != 4:
        raise ValueError("%s expects a rank-4 NHWC tensor, got shape %s" % (what, tuple(t.shape)))
    return tuple(int(v) for v in t.shape)


def conv2d(tensor, filt, post=_lib.POST_NONE, clip_max=0.0):
    x = as_device_tensor(tensor)
    n, h, w, cin = _nhwc(x, "conv2d")
    f = filter_on_device(filt, x.device)
    if f.dim() != 4 or f.shape[0] != f.shape[1] or f.shape[2] != cin:
        raise ValueError("filter of shape %s does not match input with %d channels" % (tuple(f.shape), cin))
    k, cout = int(f.shape[0]), int(f.shape[3])
    out = torch.empty((n, h, w, cout), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_conv2d(ptr(x), n, h, w, cin, ptr(f), k, cout, post, clip_max, ptr(out),
                                            stream_ptr()), "silent_conv2d")
    return out


def regulate(tensor, blur, value, root):
    x = as_device_tensor(tensor)
    n, h, w, c = _nhwc(x, "regulate_tensor")
    f = filter_on_device(blur, x.device)
    if f.dim() != 4 or f.shape[0] != f.shape[1] or f.shape[2] != c or f.shape[3] != c:
        raise ValueError("blur of shape %s does not match a %d-channel input" % (tuple(f.shape), c))
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_regulate(ptr(x), n, h, w, c, ptr(f), int(f.shape[0]), value, root, ptr(out),
                                              stream_ptr()), "silent_regulate")
    return out


def pad_inwards(tensor, top, bottom, left, right):
    x = as_device_tensor(tensor)
    n, h, w, c = _nhwc(x, "pad_inwards")
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_pad_inwards(ptr(x), n, h, w, c, top, bottom, left, right, ptr(out), stream_ptr()),
                   "silent_pad_inwards")
    return out


def value_from_color(tensor):
    x = as_device_tensor(tensor)
    n, h, w, c = _nhwc(x, "get_value_from_color")
    out = torch.empty((n, h, w, 1), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_value_from_color(ptr(x), n, h, w, c, ptr(out), stream_ptr()),
                   "silent_value_from_color")
    return out


def _selection_workspace(n, h, w, device):
    nbytes = _lib.lib().silent_selection_workspace_bytes(n, h, w)
    return torch.empty(nbytes, dtype=torch.uint8, device=device), nbytes


def max_value_indices_region(value, region_h, region_w, capacity=None):
    v = as_device_tensor(value)
    n, h, w, c = _nhwc(v, "max_value_indices_region")
    if c != 1:
        raise ValueError("value tensor must have one channel")
    ws, nbytes = _selection_workspace(n, h, w, v.device)
    cap = int(capacity) if capacity is not None else max(64 * n, 1024)
    count = torch.zeros(1, dtype=torch.int64, device=v.device)
    with torch.cuda.device(v.device):
        while True:
            pts = torch.empty((cap, 4), dtype=torch.int64, device=v.device)
            _lib.check(_lib.lib().silent_max_value_indices_region(ptr(v), n, h, w, region_h, region_w, ptr(pts), cap,
                                                                  ptr(count), ptr(ws), nbytes, stream_ptr()),
                       "silent_max_value_indices_region")
            total = int(count.item())   # tf.where has a data-dependent shape: one sync, like a session.run fetch
            if total <= cap or capacity is not None:
                return pts[:min(total, cap)]
            cap = total


def peak_percent(top_percent):
    """``top_percent`` of the peak emit as a float in [0, 1]; anything else (a bool, a non-number, NaN, a value out of
    range) raises ValueError."""
    if isinstance(top_percent, (bool, np.bool_)) or not isinstance(top_percent, numbers.Real):
        raise ValueError("peaks (top_percent) must be a real number in [0, 1], got %r" % (top_percent,))
    p = float(top_percent)
    if not 0.0 <= p <= 1.0:
        raise ValueError("peaks (top_percent) must be in [0, 1], got %r" % (top_percent,))
    return p


def peak_points(value, top_percent, capacity=None):
    """``silent_peak_points``: int64 rows ``(level, y, x, 0)`` of every 3 x 3 local maximum of ``value``
    ``[n, h, w, 1]`` that is > 0 and >= its level's top-percent threshold, in row-major order. Without ``capacity``
    every point is returned (one host synchronisation, and a second emit when they exceed the first buffer); with it, at
    most ``capacity`` rows."""
    p = peak_percent(top_percent)
    v = as_device_tensor(value)
    n, h, w, c = _nhwc(v, "peak_points")
    if c != 1:
        raise ValueError("value tensor must have one channel")
    ws, nbytes = _selection_workspace(n, h, w, v.device)
    cap = int(capacity) if capacity is not None else max(64 * n, 1024)
    count = torch.zeros(1, dtype=torch.int64, device=v.device)
    with torch.cuda.device(v.device):
        while True:
            pts = torch.empty((cap, 4), dtype=torch.int64, device=v.device)
            _lib.check(_lib.lib().silent_peak_points(ptr(v), n, h, w, p, ptr(pts), cap, ptr(count), ptr(ws), nbytes,
                                                     stream_ptr()), "silent_peak_points")
            total = int(count.item())
            if total <= cap or capacity is not None:
                return pts[:min(total, cap)]
            cap = total


def plan_peak_points(plan, batch, top_percent, points, count):
    """``silent_plan_peak_points``: the peak emit on the plan's own gray of its latest pipeline call (``batch`` frames)
    into ``points`` ``[capacity, 4]`` int64 and the int64 device scalar ``count``; no host synchronisation."""
    with torch.cuda.device(points.device):
        _lib.check(_lib.lib().silent_plan_peak_points(plan.handle, int(batch), float(top_percent), ptr(points),
                                                      int(points.shape[0]), ptr(count), stream_ptr()),
                   "silent_plan_peak_points")


def top_value_points(color, value, top_percent):
    x = as_device_tensor(color)
    v = as_device_tensor(value)
    n, h, w, c = _nhwc(x, "top_value_points")
    if tuple(v.shape) != (n, h, w, 1):
        raise ValueError("value tensor shape %s does not match colour tensor %s" % (tuple(v.shape), tuple(x.shape)))
    ws, nbytes = _selection_workspace(n, h, w, x.device)
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_top_value_points(ptr(x), ptr(v), n, h, w, c, float(top_percent), ptr(out), ptr(ws),
                                                      nbytes, stream_ptr()), "silent_top_value_points")
    return out


def get_centroids(value, region_h, region_w, want_distance=True):
    """-> (centroids [n,h,w,1] or None, total_pool [n,oh,ow,1], corrected_pool [n,oh,ow,2])."""
    v = as_device_tensor(value)
    n, h, w, c = _nhwc(v, "get_centroids")
    if c != 1:
        raise ValueError("value tensor must have one channel")
    oh, ow = -(-h // region_h), -(-w // region_w)
    corrected = torch.empty((n, oh, ow, 2), dtype=torch.float32, device=v.device)
    total = torch.empty((n, oh, ow, 1), dtype=torch.float32, device=v.device)
    cent = torch.empty((n, h, w, 1), dtype=torch.float32, device=v.device) if want_distance else None
    with torch.cuda.device(v.device):
        _lib.check(_lib.lib().silent_get_centroids(ptr(v), n, h, w, region_h, region_w, ptr(corrected), ptr(total),
                                                   ptr(cent), stream_ptr()), "silent_get_centroids")
    return cent, total, corrected


def resize_nearest(tensor, out_h, out_w):
    x = as_device_tensor(tensor)
    n, h, w, c = _nhwc(x, "resize_nearest_neighbor")
    out = torch.empty((n, int(out_h), int(out_w), c), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_resize_nearest(ptr(x), n, h, w, c, int(out_h), int(out_w), ptr(out), stream_ptr()),
                   "silent_resize_nearest")
    return out


def boosting(inp, energy, exhaustion_max, excitation_max, recovery_mode):
    """Updates ``energy`` (CUDA float32, same shape as ``inp``) in place; returns has_fired."""
    x = as_device_tensor(inp)
    n, h, w, c = _nhwc(x, "get_boosting")
    if c != 1 or tuple(energy.shape) != tuple(x.shape) or not energy.is_cuda or energy.dtype != torch.float32 \
            or not energy.is_contiguous():
        raise ValueError("exhaustion tensor must be a contiguous CUDA float32 tensor shaped like the one-channel input")
    fired = torch.empty_like(x)
    scratch = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_get_boosting(ptr(x), ptr(energy), n, h, w, float(exhaustion_max),
                                                  float(excitation_max), int(recovery_mode), ptr(fired), ptr(scratch),
                                                  stream_ptr()), "silent_get_boosting")
    return fired


def pointwise(x, kind, y=None):
    x = as_device_tensor(x)
    y = as_device_tensor(y) if y is not None else None
    if y is not None and y.shape != x.shape:
        raise ValueError("pointwise product needs equal shapes, got %s and %s" % (tuple(x.shape), tuple(y.shape)))
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_pointwise(ptr(x), ptr(y), x.numel(), int(kind), ptr(out), stream_ptr()),
                   "silent_pointwise")
    return out


def display_tensors(gray, energy, region_h, region_w, half_h, half_w, exhaustion_max, excitation_max, recovery_mode):
    """The display chain after ``gray_line_end_tensor`` in two launches (``silent_display_tensors``): returns
    ``(255 - centroids * 255, 255 - centroids2 * 255, fired * importance * 255 [.., 3], energy display [.., 3])`` and
    updates ``energy`` in place."""
    g = as_device_tensor(gray)
    n, h, w, c = _nhwc(g, "display_tensors")
    oh, ow = -(-h // region_h), -(-w // region_w)
    if c != 1 or tuple(energy.shape) != (n, oh, ow, 1) or not energy.is_cuda or energy.dtype != torch.float32 \
            or not energy.is_contiguous():
        raise ValueError("display_tensors needs a one-channel gray tensor and a contiguous CUDA float32 energy tensor "
                         "[n, ceil(h / region_h), ceil(w / region_w), 1]")
    dev = g.device
    cent = torch.empty((n, h, w, 1), dtype=torch.float32, device=dev)
    cent2 = torch.empty((n, int(half_h), int(half_w), 1), dtype=torch.float32, device=dev)
    fired = torch.empty((n, oh, ow, 3), dtype=torch.float32, device=dev)
    update = torch.empty((n, oh, ow, 3), dtype=torch.float32, device=dev)
    scratch = torch.empty((2 * n * oh * ow,), dtype=torch.float32, device=dev)
    normer = 255.0 / (exhaustion_max + excitation_max)                                   # boosting.py:37-38
    centerer = (excitation_max / (exhaustion_max + excitation_max)) * 255.0
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().silent_display_tensors(
            ptr(g), n, h, w, int(region_h), int(region_w), int(half_h), int(half_w), ptr(energy), float(exhaustion_max),
            float(excitation_max), int(recovery_mode), float(normer), float(centerer), ptr(cent), ptr(cent2), ptr(fired),
            ptr(update), ptr(scratch), stream_ptr()), "silent_display_tensors")
    return cent, cent2, fired, update


def display_sequence(gray, energy, steps, region_h, region_w, half_h, half_w, exhaustion_max, excitation_max,
                     recovery_mode):
    """``display_tensors`` over a clip (``silent_display_sequence``): ``gray`` ``[steps * n, h, w, 1]`` is time-major
    (image ``t * n + e`` is step t of slice e of ``energy`` ``[n, oh, ow, 1]``). Returns the four display tensors over
    all ``steps * n`` images, equal to ``steps`` successive ``display_tensors`` calls, and leaves ``energy`` where the
    last of them would."""
    g = as_device_tensor(gray)
    total, h, w, c = _nhwc(g, "display_sequence")
    steps = int(steps)
    n = total // steps if steps > 0 else 0
    oh, ow = -(-h // region_h), -(-w // region_w)
    if c != 1 or n <= 0 or total != steps * n or tuple(energy.shape) != (n, oh, ow, 1) or not energy.is_cuda \
            or energy.dtype != torch.float32 or not energy.is_contiguous():
        raise ValueError("display_sequence needs a one-channel gray tensor of steps * n images and a contiguous CUDA "
                         "float32 energy tensor [n, ceil(h / region_h), ceil(w / region_w), 1]")
    dev = g.device
    cent = torch.empty((total, h, w, 1), dtype=torch.float32, device=dev)
    cent2 = torch.empty((total, int(half_h), int(half_w), 1), dtype=torch.float32, device=dev)
    fired = torch.empty((total, oh, ow, 3), dtype=torch.float32, device=dev)
    update = torch.empty((total, oh, ow, 3), dtype=torch.float32, device=dev)
    nbytes = display_sequence_scratch_bytes(steps, n, h, w, region_h, region_w)
    scratch = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    normer = 255.0 / (exhaustion_max + excitation_max)                                   # boosting.py:37-38
    centerer = (excitation_max / (exhaustion_max + excitation_max)) * 255.0
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().silent_display_sequence(
            ptr(g), steps, n, h, w, int(region_h), int(region_w), int(half_h), int(half_w), ptr(energy),
            float(exhaustion_max), float(excitation_max), int(recovery_mode), float(normer), float(centerer), ptr(cent),
            ptr(cent2), ptr(fired), ptr(update), ptr(scratch), nbytes, stream_ptr()), "silent_display_sequence")
    return cent, cent2, fired, update


def display_sequence_scratch_bytes(steps, n, h, w, region_h, region_w):
    """Bytes of device scratch ``display_sequence`` allocates for one call."""
    return int(_lib.lib().silent_display_sequence_scratch_bytes(int(steps), int(n), int(h), int(w), int(region_h),
                                                                int(region_w)))


# frame layouts LineEndPipeline(frame_format=...) takes: interleaved [H, W, 3] BGR, or NV12 (include/silent_b200.h)
FRAME_FORMATS = ("bgr", "nv12")


def nv12_frame_hw(shape, dtype, ranks=(2, 3), what="NV12 frames"):
    """``(H, W)`` of NV12 frames of ``shape`` (a uint8 ``[H * 3 / 2, W]`` array per frame, in an array of one of the
    ``ranks``); ``ValueError`` for another dtype, rank or an odd frame size."""
    if dtype not in (np.uint8, torch.uint8):
        raise ValueError("%s are uint8, got %s" % (what, dtype))
    shape = tuple(int(v) for v in shape)
    if len(shape) not in ranks or min(shape, default=0) < 1:
        raise ValueError("%s need rank %s with no empty axis ([..., H * 3 / 2, W]), got shape %s"
                         % (what, " or ".join(str(r) for r in ranks), shape))
    rows, w = shape[-2:]
    if rows % 3 or w % 2:
        raise ValueError("%s need even height and width: %d rows of %d is not [H * 3 / 2, W] with H, W even"
                         % (what, rows, w))
    return 2 * rows // 3, w


def nv12_to_bgr(frames):
    """``silent_nv12_to_bgr``: NV12 frames ``[B, H * 3 / 2, W]`` (or one ``[H * 3 / 2, W]``), uint8, on the GPU ->
    contiguous BGR ``[B, H, W, 3]`` uint8 on the same device, bit for bit ``cv2.cvtColor(frame, COLOR_YUV2BGR_NV12)``."""
    h, w = nv12_frame_hw(frames.shape, frames.dtype)
    x = as_device_tensor(frames, torch.uint8)
    x = x if x.dim() == 3 else x.unsqueeze(0)
    b = int(x.shape[0])
    out = torch.empty((b, h, w, 3), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_nv12_to_bgr(ptr(x), b, h, w, ptr(out), stream_ptr()), "silent_nv12_to_bgr")
    return out


# output dtypes of the fused stacks: float32, or binary16 through the entry points named <symbol>_f16
OUT_DTYPES = (torch.float32, torch.float16)


def _stack(symbol, noun, pyramid, weights, channels, want_orient, want_line_end, want_gray, out_dtype):
    if out_dtype not in OUT_DTYPES:
        raise ValueError("%s writes float32 or float16 outputs, not %s" % (noun, out_dtype))
    x = as_device_tensor(pyramid)
    n, h, w, c = _nhwc(x, symbol[len("silent_"):])
    if c != 3:
        raise ValueError("%s needs 3-channel pyramids" % noun)
    if out_dtype == torch.float16:
        symbol += "_f16"
    mk = lambda ch, dt: torch.empty((n, h, w, ch), dtype=dt, device=x.device)  # noqa: E731
    orient = mk(channels, out_dtype) if want_orient else None
    line_end = mk(channels, out_dtype) if want_line_end else None
    gray = mk(1, torch.float32) if want_gray else None
    nbytes = _lib.lib().silent_stack_workspace_bytes(n, h, w)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(getattr(_lib.lib(), symbol)(ptr(x), n, h, w, ctypes.byref(weights), ptr(orient), ptr(line_end),
                                               ptr(gray), ptr(ws), nbytes, stream_ptr()), symbol)
    return orient, line_end, gray


def stack_fused(pyramid, weights, want_orient=True, want_line_end=True, want_gray=True, out_dtype=torch.float32):
    """The fused three-orientation stack (``silent_stack_fused``, or ``silent_stack_fused_f16`` for float16 outputs) on a
    finite NHWC pyramid: orient and padded_line_end ``[n, h, w, 3]`` of ``out_dtype``, gray ``[n, h, w, 1]`` float32."""
    return _stack("silent_stack_fused", "the fused stack", pyramid, weights, 3, want_orient, want_line_end, want_gray,
                  out_dtype)


def stack_bank(pyramid, bank, want_orient=True, want_line_end=True, want_gray=True, out_dtype=torch.float32):
    """The orientation bank's stack (``silent_stack_bank``, or ``silent_stack_bank_f16`` for float16 outputs) on a finite
    NHWC pyramid ``[n, h, w, 3]``: returns orient and padded_line_end ``[n, h, w, bank.orientations]`` of ``out_dtype``
    and gray ``[n, h, w, 1]`` float32."""
    return _stack("silent_stack_bank", "the fused orientation bank", pyramid, bank, int(bank.orientations), want_orient,
                  want_line_end, want_gray, out_dtype)


def patch_radius(radius):
    """``radius`` as an int in ``[0, PATCH_RADIUS_MAX]``, or None for None; anything else (a bool, a float, a value out
    of range) raises ValueError."""
    if radius is None:
        return None
    if isinstance(radius, bool) or not isinstance(radius, (int, np.integer)):
        raise ValueError("patch radius must be an int, got %r" % (radius,))
    if not 0 <= radius <= _lib.PATCH_RADIUS_MAX:
        raise ValueError("patch radius must be in [0, %d], got %d" % (_lib.PATCH_RADIUS_MAX, radius))
    return int(radius)


def record_values_shape(capacity, channels, radius=None):
    """Shape of the float32 ``values`` of ``capacity`` records of ``channels`` channels: ``[capacity, 1 + 2C]``, or
    ``[capacity, P, P, 1 + 2C]`` with a patch of radius ``radius`` (P = 2 * radius + 1)."""
    v = 1 + 2 * channels
    return (capacity, v) if radius is None else (capacity, 2 * radius + 1, 2 * radius + 1, v)


def check_record_buffers(batch, capacity, channels, radius, frame_offsets, frame_yx, values):
    """ValueError unless ``frame_offsets``, ``frame_yx`` and ``values`` are the int64 / float32 / float32 tensors that
    ``capacity`` records of ``batch`` frames with ``channels`` channels (and a patch of ``radius``) fill."""
    for name, t, dt, shape in (("frame_offsets", frame_offsets, torch.int64, (batch + 1,)),
                               ("frame_yx", frame_yx, torch.float32, (capacity, 2)),
                               ("values", values, torch.float32, record_values_shape(capacity, channels, radius))):
        if not isinstance(t, torch.Tensor):
            raise ValueError("%s must be %s %s, got %s" % (name, dt, shape, type(t).__name__))
        if t.dtype != dt or tuple(t.shape) != shape:
            raise ValueError("%s must be %s %s, got %s %s" % (name, dt, shape, t.dtype, tuple(t.shape)))


def point_records(plan, batch, points, count, orient, line_end, gray=None, frame_offsets=None, frame_yx=None,
                  values=None, radius=None):
    """``silent_point_records``: the records of the first ``min(count, capacity)`` rows of ``points`` ``[capacity, 4]``
    int64 (``count``: an int64 device scalar, the emit's total). ``orient`` and ``line_end`` are the call's
    ``[batch * L, h, w, C]`` outputs (float32 or float16, C = 3, 4, 8, 12 or 16); ``gray`` ``[batch * L, h, w, 1]``
    float32, or None for the plan's own gray of its latest pipeline call. Returns ``(frame_offsets [batch + 1] int64,
    frame_yx [capacity, 2] float32, values [capacity, 1 + 2C] float32)``, into the given buffers where passed; no host
    synchronisation. With an int ``radius`` (``silent_point_patches``) ``values`` is ``[capacity, P, P, 1 + 2C]``, the
    patch of side P = 2 * radius + 1 around each point, +0.0 outside the level. Shapes, dtypes, devices and the radius
    are checked first (ValueError)."""
    radius = patch_radius(radius)
    batch = int(batch)
    if batch <= 0:
        raise ValueError("point_records needs a positive batch, got %d" % batch)
    n = batch * plan.levels
    if orient.dim() != 4 or orient.shape[:3] != (n, plan.h, plan.w) or line_end.shape != orient.shape:
        raise ValueError("point_records needs orient and line_end of shape [%d, %d, %d, C], got %s and %s"
                         % (n, plan.h, plan.w, tuple(orient.shape), tuple(line_end.shape)))
    c = int(orient.shape[3])
    if c not in _lib.RECORD_CHANNELS:
        raise ValueError("point_records reads 3, 4, 8, 12 or 16 channels, got %d" % c)
    if orient.dtype not in OUT_DTYPES or line_end.dtype != orient.dtype:
        raise ValueError("orient and line_end must both be float32 or both float16, got %s and %s"
                         % (orient.dtype, line_end.dtype))
    if points.dim() != 2 or points.shape[1] != 4 or points.dtype != torch.int64:
        raise ValueError("points must be int64 [capacity, 4], got %s %s" % (points.dtype, tuple(points.shape)))
    cap = int(points.shape[0])
    if count.dtype != torch.int64 or count.numel() < 1:
        raise ValueError("count must be an int64 tensor of at least one element")
    if gray is not None and (gray.dtype != torch.float32 or tuple(gray.shape) != (n, plan.h, plan.w, 1)):
        raise ValueError("gray must be float32 [%d, %d, %d, 1], got %s %s" % (n, plan.h, plan.w, gray.dtype,
                                                                            tuple(gray.shape)))
    dev = points.device
    mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)  # noqa: E731
    frame_offsets = mk((batch + 1,), torch.int64) if frame_offsets is None else frame_offsets
    frame_yx = mk((cap, 2), torch.float32) if frame_yx is None else frame_yx
    values = mk(record_values_shape(cap, c, radius), torch.float32) if values is None else values
    check_record_buffers(batch, cap, c, radius, frame_offsets, frame_yx, values)
    tensors = [points, count, orient, line_end, frame_offsets, frame_yx, values] + ([gray] if gray is not None else [])
    if any(not t.is_cuda or t.device != dev or not t.is_contiguous() for t in tensors):
        raise ValueError("point_records needs contiguous CUDA tensors on one device")
    half = int(orient.dtype == torch.float16)
    with torch.cuda.device(dev):
        if radius is None:
            _lib.check(_lib.lib().silent_point_records(
                plan.handle, batch, ptr(points), ptr(count), cap, ptr(orient), ptr(line_end), c, half, ptr(gray),
                ptr(frame_offsets), ptr(frame_yx), ptr(values), stream_ptr()), "silent_point_records")
        else:
            _lib.check(_lib.lib().silent_point_patches(
                plan.handle, batch, ptr(points), ptr(count), cap, ptr(orient), ptr(line_end), c, half, ptr(gray),
                radius, ptr(frame_offsets), ptr(frame_yx), ptr(values), stream_ptr()), "silent_point_patches")
    return frame_offsets, frame_yx, values


def match_radius(radius):
    """``radius`` of the match search window as an int in ``[0, 2^31 - 1]``; anything else (a bool, a float, a str, a
    negative value) raises ValueError."""
    if isinstance(radius, (bool, np.bool_)) or not isinstance(radius, (int, np.integer)):
        raise ValueError("search radius must be an int, got %r" % (radius,))
    if not 0 <= radius <= 2 ** 31 - 1:
        raise ValueError("search radius must be in [0, 2^31 - 1], got %d" % radius)
    return int(radius)


def match_ratio(max_ratio):
    """``max_ratio`` of the match ratio test as a float in (0, 1]; anything else (a bool, a non-number, NaN, a value out
    of range) raises ValueError."""
    if isinstance(max_ratio, (bool, np.bool_)) or not isinstance(max_ratio, numbers.Real):
        raise ValueError("max_ratio must be a real number in (0, 1], got %r" % (max_ratio,))
    m = float(max_ratio)
    if not 0.0 < m <= 1.0 or not 0.0 < float(np.float32(m)) <= 1.0:
        raise ValueError("max_ratio must be in (0, 1], got %r" % (max_ratio,))
    return m


def match_points(points, count, values, levels, search_radius, max_ratio=1.0, next=None, prev=None, distance=None):
    """``silent_match_points``: mutual nearest descriptors between consecutive frames. ``points`` ``[capacity, 4]``
    int64 rows ``(level, y, x, 0)`` sorted by (level, y, x), level = frame * ``levels`` + l; ``count`` an int64 device
    scalar (the rows used are the first ``clamp(count, 0, capacity)``); ``values`` float32 ``[capacity, ...]``, each
    row's descriptor of E = the product of the trailing shape elements. Returns ``(next, prev, distance)``: int64, int64
    and float32 ``[capacity]`` (see ``pipeline.PointMatches``), into the given buffers where passed; no host
    synchronisation. Shapes, dtypes, devices, contiguity and the arguments are checked first (ValueError)."""
    radius = match_radius(search_radius)
    ratio = match_ratio(max_ratio)
    if isinstance(levels, (bool, np.bool_)) or not isinstance(levels, (int, np.integer)) or not 1 <= levels < 2 ** 31:
        raise ValueError("match_points needs levels as an int >= 1, got %r" % (levels,))
    for name, t in (("points", points), ("count", count), ("values", values)):
        if not isinstance(t, torch.Tensor):
            raise ValueError("%s must be a torch.Tensor, got %s" % (name, type(t).__name__))
    if points.dim() != 2 or points.shape[1] != 4 or points.dtype != torch.int64:
        raise ValueError("points must be int64 [capacity, 4], got %s %s" % (points.dtype, tuple(points.shape)))
    cap = int(points.shape[0])
    if count.dtype != torch.int64 or count.numel() < 1:
        raise ValueError("count must be an int64 tensor of at least one element")
    if values.dtype != torch.float32 or values.dim() < 1 or int(values.shape[0]) != cap:
        raise ValueError("values must be float32 [%d, ...], got %s %s" % (cap, values.dtype, tuple(values.shape)))
    elems = int(np.prod(values.shape[1:], dtype=np.int64))
    if elems < 1:
        raise ValueError("values must hold at least one element per row, got %s" % (tuple(values.shape),))
    dev = points.device
    mk = lambda dt: torch.empty((cap,), dtype=dt, device=dev)  # noqa: E731
    next = mk(torch.int64) if next is None else next
    prev = mk(torch.int64) if prev is None else prev
    distance = mk(torch.float32) if distance is None else distance
    for name, t, dt in (("next", next, torch.int64), ("prev", prev, torch.int64), ("distance", distance, torch.float32)):
        if not isinstance(t, torch.Tensor) or t.dtype != dt or tuple(t.shape) != (cap,):
            raise ValueError("%s must be %s [%d], got %s" % (name, dt, cap, getattr(t, "dtype", type(t).__name__)))
    tensors = (points, count, values, next, prev, distance)
    if any(not t.is_cuda or t.device != dev or not t.is_contiguous() for t in tensors):
        raise ValueError("match_points needs contiguous CUDA tensors on one device")
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().silent_match_points(
            ptr(points), ptr(count), cap, ptr(values), elems, int(levels), radius, ratio, ptr(next), ptr(prev),
            ptr(distance), stream_ptr()), "silent_match_points")
    return next, prev, distance


def motion_args(threshold, hypotheses, seed):
    """``(threshold, hypotheses, seed)`` of ``estimate_motion`` as (float, int, int): ``threshold`` a real number whose
    float32 value is finite and > 0 (frame pixels), ``hypotheses`` an int in ``[1, MOTION_HYPOTHESES_MAX]``, ``seed`` an
    int in ``[0, 2^64)``; anything else (a bool, a non-number, NaN, a value out of range) raises ValueError."""
    if isinstance(threshold, (bool, np.bool_)) or not isinstance(threshold, numbers.Real):
        raise ValueError("threshold must be a real number > 0, got %r" % (threshold,))
    t = float(threshold)
    with np.errstate(over="ignore"):
        t32 = float(np.float32(t))
    if not (math.isfinite(t32) and t32 > 0.0):
        raise ValueError("threshold must be finite and > 0 in float32, got %r" % (threshold,))
    if isinstance(hypotheses, (bool, np.bool_)) or not isinstance(hypotheses, (int, np.integer)) \
            or not 1 <= hypotheses <= _lib.MOTION_HYPOTHESES_MAX:
        raise ValueError("hypotheses must be an int in [1, %d], got %r" % (_lib.MOTION_HYPOTHESES_MAX, hypotheses))
    if isinstance(seed, (bool, np.bool_)) or not isinstance(seed, (int, np.integer)) or not 0 <= seed < 2 ** 64:
        raise ValueError("seed must be an int in [0, 2^64), got %r" % (seed,))
    return t, int(hypotheses), int(seed)


def motion_workspace_bytes(capacity):
    """Bytes of the ``estimate_motion`` workspace for ``capacity`` rows (``silent_motion_workspace_bytes``)."""
    return int(_lib.lib().silent_motion_workspace_bytes(int(capacity)))


def estimate_motion(frame_offsets, frame_yx, next, count, hypotheses, threshold, seed=0, transform=None,
                    inlier_count=None, matched=None, inlier=None, workspace=None):
    """``silent_estimate_motion``: a robust affine map per pair of consecutive frames from the matches. ``frame_offsets``
    int64 ``[B + 1]`` and ``frame_yx`` float32 ``[capacity, 2]`` as ``PointRecords`` holds them, ``next`` int64
    ``[capacity]`` as ``PointMatches`` holds it, ``count`` an int64 device scalar (the rows used are the first
    ``clamp(count, 0, capacity)``). Returns ``(transform, inlier_count, matched, inlier)``: float64 ``[B - 1, 2, 3]``,
    int64 ``[B - 1]``, int64 ``[B - 1]`` and uint8 ``[capacity]`` (see ``pipeline.PointMotion``), into the given buffers
    where passed; ``workspace`` a uint8 tensor of at least ``motion_workspace_bytes(capacity)`` bytes. No host
    synchronisation. Shapes, dtypes, devices, contiguity and the arguments are checked first (ValueError)."""
    threshold, hypotheses, seed = motion_args(threshold, hypotheses, seed)
    for name, t in (("frame_offsets", frame_offsets), ("frame_yx", frame_yx), ("next", next), ("count", count)):
        if not isinstance(t, torch.Tensor):
            raise ValueError("%s must be a torch.Tensor, got %s" % (name, type(t).__name__))
    if frame_offsets.dim() != 1 or frame_offsets.shape[0] < 2 or frame_offsets.dtype != torch.int64:
        raise ValueError("frame_offsets must be int64 [B + 1] with B >= 1, got %s %s"
                         % (frame_offsets.dtype, tuple(frame_offsets.shape)))
    batch = int(frame_offsets.shape[0]) - 1
    if batch > 2 ** 31 - 1:
        raise ValueError("estimate_motion takes at most 2^31 - 1 frames, got %d" % batch)
    if frame_yx.dim() != 2 or frame_yx.shape[1] != 2 or frame_yx.dtype != torch.float32:
        raise ValueError("frame_yx must be float32 [capacity, 2], got %s %s" % (frame_yx.dtype, tuple(frame_yx.shape)))
    cap = int(frame_yx.shape[0])
    if next.dtype != torch.int64 or tuple(next.shape) != (cap,):
        raise ValueError("next must be int64 [%d], got %s %s" % (cap, next.dtype, tuple(next.shape)))
    if count.dtype != torch.int64 or count.numel() < 1:
        raise ValueError("count must be an int64 tensor of at least one element")
    dev = frame_yx.device
    pairs = batch - 1
    transform = torch.empty((pairs, 2, 3), dtype=torch.float64, device=dev) if transform is None else transform
    inlier_count = torch.empty((pairs,), dtype=torch.int64, device=dev) if inlier_count is None else inlier_count
    matched = torch.empty((pairs,), dtype=torch.int64, device=dev) if matched is None else matched
    inlier = torch.empty((cap,), dtype=torch.uint8, device=dev) if inlier is None else inlier
    need = motion_workspace_bytes(cap)
    workspace = torch.empty((max(need, 1),), dtype=torch.uint8, device=dev) if workspace is None else workspace
    for name, t, dt, shape in (("transform", transform, torch.float64, (pairs, 2, 3)),
                               ("inlier_count", inlier_count, torch.int64, (pairs,)),
                               ("matched", matched, torch.int64, (pairs,)), ("inlier", inlier, torch.uint8, (cap,))):
        if not isinstance(t, torch.Tensor) or t.dtype != dt or tuple(t.shape) != shape:
            raise ValueError("%s must be %s %s, got %s %s" % (name, dt, shape, getattr(t, "dtype", type(t).__name__),
                                                               tuple(getattr(t, "shape", ()))))
    if not isinstance(workspace, torch.Tensor) or workspace.dtype != torch.uint8 or workspace.dim() != 1 \
            or workspace.numel() < need:
        raise ValueError("workspace must be a uint8 tensor of at least %d bytes" % need)
    tensors = (frame_offsets, frame_yx, next, count, transform, inlier_count, matched, inlier, workspace)
    if any(not t.is_cuda or t.device != dev or not t.is_contiguous() for t in tensors):
        raise ValueError("estimate_motion needs contiguous CUDA tensors on one device")
    if workspace.data_ptr() % 16:
        raise ValueError("workspace must be 16-byte aligned")
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().silent_estimate_motion(
            ptr(frame_offsets), ptr(frame_yx), ptr(next), ptr(count), cap, batch, hypotheses, threshold, seed,
            ptr(workspace), workspace.numel(), ptr(transform), ptr(inlier_count), ptr(matched), ptr(inlier),
            stream_ptr()), "silent_estimate_motion")
        if cap == 0 or batch == 1:   # the library launches nothing then: no pair has a correspondence
            transform.fill_(float("nan"))
            inlier_count.zero_()
            matched.zero_()
            inlier.zero_()
    return transform, inlier_count, matched, inlier
