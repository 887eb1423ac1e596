"""Device-side operator implementations over the C ABI. torch supplies device memory and streams only.

Tensors are contiguous float32 NHWC ``[levels, h, w, C]`` on a CUDA device (the reference's placeholder layout,
``recognition_testing.py:62``); numpy inputs are uploaded to the current CUDA device.
"""
import ctypes
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


def stack_fused(pyramid, weights, want_orient=True, want_line_end=True, want_gray=True):
    x = as_device_tensor(pyramid)
    n, h, w, c = _nhwc(x, "stack_fused")
    if c != 3:
        raise ValueError("the fused stack needs 3-channel pyramids")
    mk = lambda ch: torch.empty((n, h, w, ch), dtype=torch.float32, device=x.device)  # noqa: E731
    orient = mk(3) if want_orient else None
    line_end = mk(3) if want_line_end else None
    gray = mk(1) if want_gray else None
    nbytes = _lib.lib().silent_stack_workspace_bytes(n, h, w)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_stack_fused(ptr(x), n, h, w, ctypes.byref(weights), ptr(orient), ptr(line_end),
                                                 ptr(gray), ptr(ws), nbytes, stream_ptr()), "silent_stack_fused")
    return orient, line_end, gray


def stack_bank(pyramid, bank, want_orient=True, want_line_end=True, want_gray=True):
    """The orientation bank's stack (``silent_stack_bank``) on a finite NHWC pyramid ``[n, h, w, 3]``: returns orient and
    padded_line_end ``[n, h, w, bank.orientations]`` and gray ``[n, h, w, 1]``."""
    x = as_device_tensor(pyramid)
    n, h, w, c = _nhwc(x, "stack_bank")
    if c != 3:
        raise ValueError("the fused orientation bank needs 3-channel pyramids")
    nb = int(bank.orientations)
    mk = lambda ch: torch.empty((n, h, w, ch), dtype=torch.float32, device=x.device)  # noqa: E731
    orient = mk(nb) if want_orient else None
    line_end = mk(nb) if want_line_end else None
    gray = mk(1) if want_gray else None
    nbytes = _lib.lib().silent_stack_workspace_bytes(n, h, w)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().silent_stack_bank(ptr(x), n, h, w, ctypes.byref(bank), ptr(orient), ptr(line_end),
                                                ptr(gray), ptr(ws), nbytes, stream_ptr()), "silent_stack_bank")
    return orient, line_end, gray
