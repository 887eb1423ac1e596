"""Which operators, fused stacks and C entry points every ``LineEndPipeline`` entry point reaches, traced on the CPU.

The leaves the pipeline calls are replaced by recorders: the ``_ops`` operators and fused stacks, the pyramid builder,
the ``silent_pipeline_run*`` C entry points, the plan cache, page-locked staging and the stream. Each entry point is
swept over orientation counts, frame formats, frame dtypes, channel counts, row widths, blur sizes, output dtypes and
finite / non-finite inputs, and its trace (the calls in order, the float32 bytes of every filter, the packed weights,
batch, points capacity, synchronisations and the shapes it returns) must equal the one stored in
``golden/pipeline_routes.json.gz`` (each distinct trace once, then the index of every case's trace). A failure shows
the first case that moved, with both traces. When a route changes on purpose, rewrite that file with
``python tests/test_pipeline_routes.py --write``.
"""
import contextlib
import ctypes
import functools
import gzip
import hashlib
import importlib
import itertools
import json
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")

HERE = os.path.dirname(os.path.abspath(__file__))
if os.path.dirname(HERE) not in sys.path:
    sys.path.insert(0, os.path.dirname(HERE))
from pysilent_b200 import _lib, _ops, pipeline  # noqa: E402
from pysilent_b200.pipeline import LineEndPipeline  # noqa: E402
from pysilent_b200.recognition_testing import LineEndDisplayer  # noqa: E402

from_image = importlib.import_module("pysilent_b200.util.zoom.from_image")   # the package exports a function of that name

GOLDEN = os.path.join(HERE, "golden", "pipeline_routes.json.gz")
ORIENTATIONS = (None, 1, 2, 3, 4, 5, 6, 7, 8, 12, 16)
LEVELS = 2          # levels of every fake plan and pyramid
EMITTED = 5         # feature points every fake C call reports (more than the capacity of 3 some cases ask for)
SIZE = (24, 16)     # output_size (w, h): region windows of 8 x 12
H = 24              # frame height. Widths 32 and 34: 3-channel rows of 96 and 102 bytes, 4-channel rows of 128 and 136
BATCH = 2
# (format, dtype, channels, width, finite)
FRAME_KINDS = ([("bgr", np.uint8, c, w, True) for c in (3, 4) for w in (32, 34)]
               + [("bgr", np.float32, c, w, finite) for c in (3, 4) for w in (32, 34) for finite in (True, False)]
               + [("nv12", np.uint8, 3, w, True) for w in (32, 34)])


def _digest(buf):
    return hashlib.sha1(bytes(buf)).hexdigest()[:12]


def _f32(a):
    a = np.ascontiguousarray(np.asarray(a), dtype=np.float32)
    return "%s:%s" % (_digest(a.tobytes()), "x".join(str(v) for v in a.shape))


def _shape(t):
    return "x".join(str(int(v)) for v in t.shape)


def _dt(dtype):
    return str(dtype).replace("torch.", "")


def _summary(x, named):
    if id(x) in named:
        return named[id(x)]
    if x is None:
        return "None"
    if isinstance(x, torch.Tensor):
        return "tensor %s %s" % (_shape(x), _dt(x.dtype))
    if isinstance(x, np.ndarray):
        return "array %s %s" % (_shape(x), x.dtype)
    return "[%s]" % ", ".join(_summary(v, named) for v in x)


class Tracer:
    """Installs the recorders with ``mp`` (a ``pytest.MonkeyPatch``); ``log`` is the trace of the calls since."""

    def __init__(self, mp):
        self.log = []
        rec = self.rec
        real_fused_input_ok = _ops.fused_input_ok

        def as_device_tensor(t, dtype=torch.float32):
            if isinstance(t, np.ndarray):
                t = torch.from_numpy(np.ascontiguousarray(t))
            rec("as_device_tensor", _shape(t), _dt(t.dtype), _dt(dtype))
            return t.to(dtype).contiguous()

        def fused_input_ok(x):
            ok = real_fused_input_ok(x)
            rec("fused_input_ok", _shape(x), ok)
            return ok

        def conv2d(x, filt, post=_lib.POST_NONE, clip_max=0.0):
            rec("conv2d", _shape(x), _f32(filt), post, clip_max)
            return torch.zeros(tuple(x.shape[:3]) + (np.shape(filt)[3],))

        def regulate(x, blur, value, root):
            rec("regulate", _shape(x), _f32(blur), value, root)
            return torch.zeros_like(x)

        def pad_inwards(x, top, bottom, left, right):
            rec("pad_inwards", _shape(x), top, bottom, left, right)
            return torch.zeros_like(x)

        def value_from_color(x):
            rec("value_from_color", _shape(x))
            return torch.zeros(tuple(x.shape[:3]) + (1,))

        def max_value_indices_region(v, region_h, region_w, capacity=None):
            rec("max_value_indices_region", _shape(v), region_h, region_w, capacity)
            return torch.zeros((EMITTED, 4), dtype=torch.int64)

        def stack(name, channels):
            def run(x, weights, want_orient=True, want_line_end=True, want_gray=True, out_dtype=torch.float32):
                rec(name, _shape(x), _digest(weights), want_orient, want_line_end, want_gray, _dt(out_dtype))
                n, h, w = x.shape[:3]
                c = channels(weights)
                return (torch.zeros((n, h, w, c), dtype=out_dtype), torch.zeros((n, h, w, c), dtype=out_dtype),
                        torch.zeros((n, h, w, 1)))
            return run

        def nv12_to_bgr(frames):
            h, w = _ops.nv12_frame_hw(frames.shape, frames.dtype)
            rec("nv12_to_bgr", _shape(frames), _dt(frames.dtype))
            return torch.zeros((frames.shape[0] if frames.dim() == 3 else 1, h, w, 3), dtype=torch.uint8)

        def image_to_zoom_tensor(image, num_colors, center, scale):
            rec("image_to_zoom_tensor", _shape(image), _dt(image.dtype), num_colors, tuple(center), scale)
            fill = 0.0 if bool(torch.isfinite(image.float()).all()) else float("nan")
            b = image.shape[0] if image.dim() == 4 else 1
            return torch.full((b * LEVELS, center[1], center[0], num_colors), fill)

        def display_tensors(gray, energy, region_h, region_w, half_h, half_w, *rest):
            rec("display_tensors", _shape(gray), _shape(energy), region_h, region_w, half_h, half_w, *rest)
            return _display_outputs(gray.shape[0], gray, energy, half_h, half_w)

        def display_sequence(gray, energy, steps, region_h, region_w, half_h, half_w, *rest):
            rec("display_sequence", _shape(gray), _shape(energy), steps, region_h, region_w, half_h, half_w, *rest)
            return _display_outputs(gray.shape[0], gray, energy, half_h, half_w)

        def _display_outputs(n, gray, energy, half_h, half_w):
            h, w = gray.shape[1:3]
            oh, ow = energy.shape[1:3]
            return (torch.zeros((n, h, w, 1)), torch.zeros((n, half_h, half_w, 1)), torch.zeros((n, oh, ow, 3)),
                    torch.zeros((n, oh, ow, 3)))

        class Plan:
            levels = LEVELS
            handle = ctypes.c_void_p(0)

            def __init__(self, pipe):
                self.w, self.h = pipe.output_size

            def reserve(self, batch):
                rec("reserve", batch)

        def plan(pipe, frame_shape, frame_dtype, device, frame_format="bgr"):
            rec("plan", "x".join(str(int(v)) for v in frame_shape), _dt(frame_dtype), frame_format)
            return Plan(pipe)

        class Lib:
            """The C entry points that take frames: record the call, report EMITTED points."""
            def __getattr__(self, name):
                if not name.startswith("silent_pipeline_run"):
                    raise AttributeError(name)

                def call(*args):
                    weights, batch, cap, count = args[1], args[3], args[-3], args[-2]
                    rec(name, _digest(weights._obj), "batch=%d" % batch, "cap=%d" % cap, count is not None)
                    if isinstance(count, ctypes.c_void_p):
                        ctypes.c_int64.from_address(count.value).value = EMITTED
                    elif count is not None:
                        count._obj.value = EMITTED
                    return 0
                return call

        class Stream:
            cuda_stream = 0

            def synchronize(self):
                rec("synchronize")

        def pin_memory(t, *args, **kwargs):
            rec("pin_memory", _shape(t), _dt(t.dtype))
            return t

        fakes = dict(as_device_tensor=as_device_tensor, fused_input_ok=fused_input_ok, conv2d=conv2d, regulate=regulate,
                     pad_inwards=pad_inwards, value_from_color=value_from_color,
                     max_value_indices_region=max_value_indices_region,
                     stack_fused=stack("stack_fused", lambda w: 3),
                     stack_bank=stack("stack_bank", lambda w: int(w.orientations)), nv12_to_bgr=nv12_to_bgr,
                     display_tensors=display_tensors, display_sequence=display_sequence,
                     _require_cuda=lambda: None, stream_ptr=lambda: ctypes.c_void_p(0))
        for name, fake in fakes.items():
            mp.setattr(_ops, name, fake)
        mp.setattr(from_image, "image_to_zoom_tensor", image_to_zoom_tensor)
        mp.setattr(pipeline, "image_to_zoom_tensor", image_to_zoom_tensor, raising=False)
        lib = Lib()
        mp.setattr(_lib, "lib", lambda: lib)
        mp.setattr(LineEndPipeline, "_plan", plan)
        stream = Stream()
        mp.setattr(torch.cuda, "device", lambda device: contextlib.nullcontext())
        mp.setattr(torch.cuda, "current_stream", lambda device=None: stream)
        mp.setattr(torch.Tensor, "pin_memory", pin_memory)
        # the bank generators are pure and slow: build each width once for the whole sweep
        mp.setattr(pipeline, "orientation_bank_filters", functools.lru_cache()(pipeline.orientation_bank_filters))

    def rec(self, *event):
        self.log.append(" ".join(str(e) for e in event))


def _pipe(cls, nb, blur, out_dtype, fmt="bgr"):
    p = cls(output_size=SIZE, zoom_ratio=1.5, orientations=nb, out_dtype=out_dtype, frame_format=fmt, device="cpu")
    p.blur_size = blur
    return p


def _frames(fmt, dtype, c, w, finite):
    if fmt == "nv12":
        return np.full((BATCH, H * 3 // 2, w), 128, np.uint8)
    a = np.full((BATCH, H, w, c), 100, dtype)
    if not finite:
        a[1, 5, 7, 1] = np.nan
    return a


def cases():
    """``(key, call)``: ``call()`` returns what the entry point returns and the names of the caller's buffers in it."""
    for nb, blur, od in itertools.product(ORIENTATIONS, (7, 5), (torch.float32, torch.float16)):
        cfg = "orientations=%s blur=%d %s" % (nb, blur, _dt(od))
        pipe = functools.partial(_pipe, LineEndPipeline, nb, blur, od)
        for finite in (True, False):
            pyr = np.full((BATCH * LEVELS, SIZE[1], SIZE[0], 3), 50, np.float32)
            if not finite:
                pyr[3, 4, 4, 0] = np.inf
            what = "%s %s pyramid" % (cfg, "finite" if finite else "non-finite")
            yield what + " run", lambda pyr=pyr: (pipe().run(pyr), {})
            yield what + " run want_points=False", lambda pyr=pyr: (pipe().run(pyr, want_points=False), {})
            yield what + " run_unfused", lambda pyr=pyr: (pipe().run_unfused(pyr), {})
            if nb is not None:
                yield what + " run_bank", lambda pyr=pyr: (pipe().run_bank(pyr), {})
        for fmt, dtype, c, w, finite in FRAME_KINDS:
            what = "%s %s %s C=%d W=%d %s" % (cfg, fmt, np.dtype(dtype), c, w, "finite" if finite else "non-finite")
            pipe = functools.partial(_pipe, LineEndPipeline, nb, blur, od, fmt)
            host = _frames(fmt, dtype, c, w, finite)
            frames = torch.from_numpy(host)
            yield what + " run_frames", lambda frames=frames: (pipe().run_frames(frames), {})
            yield what + " run_frames one frame", lambda frames=frames: (pipe().run_frames(frames[0]), {})
            yield (what + " run_frames want_points=False",
                   lambda frames=frames: (pipe().run_frames(frames, want_points=False), {}))
            yield (what + " run_frames points_capacity=3",
                   lambda frames=frames: (pipe().run_frames(frames, points_capacity=3), {}))

            def into_out(frames=frames):
                res_shape = (BATCH * LEVELS, SIZE[1], SIZE[0], nb or 3)
                out = (torch.zeros(res_shape, dtype=od), torch.zeros(res_shape, dtype=od),
                       torch.zeros((64, 4), dtype=torch.int64), torch.zeros(1, dtype=torch.int64))
                return pipe().run_frames(frames, out=out), {id(t): "out[%d]" % i for i, t in enumerate(out)}
            yield what + " run_frames out=", into_out
            yield what + " run_host", lambda host=host: (pipe().run_host(host), {})

            def host_into(host=host):
                np_dtype = np.float16 if od == torch.float16 else np.float32
                orient_out = np.zeros((BATCH * LEVELS, SIZE[1], SIZE[0], nb or 3), np_dtype)
                line_end_out = np.zeros_like(orient_out)
                res = pipe().run_host(host, orient_out, line_end_out, points_capacity=3)
                return res, {id(orient_out): "orient_out", id(line_end_out): "line_end_out"}
            yield what + " run_host into caller arrays, points_capacity=3", host_into
            if od == torch.float32:
                display = functools.partial(_pipe, LineEndDisplayer, nb, blur, od, fmt)
                yield what + " callback", lambda host=host: (display().callback(host[0]), {})
                yield what + " callback_clip", lambda host=host: (display().callback_clip(host), {})


def traces():
    out = {}
    with pytest.MonkeyPatch.context() as mp:
        tracer = Tracer(mp)
        for key, call in cases():
            tracer.log = []
            try:
                res, named = call()
                tracer.rec("->", _summary(res, named))
            except ValueError as exc:
                tracer.rec("ValueError", exc)
            out[key] = tracer.log
    return out


def write_golden(path=GOLDEN):
    got = traces()
    distinct = sorted(set(tuple(t) for t in got.values()))
    index = {t: i for i, t in enumerate(distinct)}
    text = '{\n"traces": [\n%s\n],\n"cases": {\n%s\n}\n}\n' % (
        ",\n".join("  " + json.dumps(list(t)) for t in distinct),
        ",\n".join("  %s: %d" % (json.dumps(k), index[tuple(t)]) for k, t in got.items()))
    with open(path, "wb") as f, gzip.GzipFile(fileobj=f, mode="wb", mtime=0) as z:   # the same bytes on every run
        z.write(text.encode())


def test_every_entry_point_reaches_the_recorded_calls():
    with gzip.open(GOLDEN, "rt") as f:
        golden = json.load(f)
    want = {key: golden["traces"][i] for key, i in golden["cases"].items()}
    got = traces()
    assert sorted(got) == sorted(want)
    moved = [key for key in want if got[key] != want[key]]
    assert not moved, "%d of %d cases take another route; first: %s\nrecorded:\n  %s\nnow:\n  %s" % (
        len(moved), len(want), moved[0], "\n  ".join(want[moved[0]]), "\n  ".join(got[moved[0]]))


def _route_table(nb, fmt, dtype, w, c, blur, colors):
    """The frame routes written out. BGR: no bank -> plan; a bank -> plan iff it has fused kernels (4, 8, 12, 16), the
    frames are uint8 with at least 3 channels, blur 7, 3 output colours and rows of a multiple of 16 bytes, else
    pyramid. NV12: plan iff the uint8 3-channel BGR frames of the same width take plan, blur 7 and 3 output colours,
    else convert."""
    fusable = blur == 7 and colors == 3
    if fmt == "nv12":
        return "plan" if fusable and _route_table(nb, "bgr", torch.uint8, w, 3, blur, colors) == "plan" else "convert"
    if nb is None:
        return "plan"
    bank_fused = nb in (4, 8, 12, 16) and dtype == torch.uint8 and c >= 3 and fusable and (w * c) % 16 == 0
    return "plan" if bank_fused else "pyramid"


def test_frame_route_table():
    spot = [((None, "bgr", torch.float32, 34, 3, 5, 3), "plan"), ((None, "nv12", torch.uint8, 34, 3, 5, 3), "convert"),
            ((None, "nv12", torch.uint8, 34, 3, 7, 1), "convert"), ((None, "nv12", torch.uint8, 34, 3, 7, 3), "plan"),
            ((12, "bgr", torch.uint8, 32, 3, 7, 3), "plan"), ((12, "bgr", torch.uint8, 34, 3, 7, 3), "pyramid"),
            ((16, "bgr", torch.uint8, 34, 4, 7, 3), "pyramid"), ((4, "bgr", torch.uint8, 36, 4, 7, 3), "plan"),
            ((8, "bgr", torch.float32, 32, 3, 7, 3), "pyramid"), ((8, "bgr", torch.uint8, 32, 3, 5, 3), "pyramid"),
            ((6, "bgr", torch.uint8, 32, 3, 7, 3), "pyramid"), ((4, "bgr", torch.uint8, 32, 1, 7, 3), "pyramid"),
            ((12, "nv12", torch.uint8, 32, 3, 7, 3), "plan"), ((12, "nv12", torch.uint8, 34, 3, 7, 3), "convert"),
            ((6, "nv12", torch.uint8, 32, 3, 7, 3), "convert")]
    for args, route in spot:
        assert _route_table(*args) == route, args
    rows = itertools.product(ORIENTATIONS, ("bgr", "nv12"), (torch.uint8, torch.float32), range(2, 68, 2), (1, 3, 4),
                             (7, 5), (3, 1))
    for nb, fmt, dtype, w, c, blur, colors in rows:
        if fmt == "nv12" and (dtype, c) != (torch.uint8, 3):
            continue
        pipe = LineEndPipeline(orientations=nb, frame_format=fmt)
        pipe.blur_size, pipe.output_colors = blur, colors
        shape = (1, H * 3 // 2, w) if fmt == "nv12" else (1, H, w, c)
        assert pipe._frame_route(nb, fmt, dtype, shape) == _route_table(nb, fmt, dtype, w, c, blur, colors), \
            (nb, fmt, dtype, w, c, blur, colors)


if __name__ == "__main__":
    if sys.argv[1:] != ["--write"]:
        sys.exit("usage: python tests/test_pipeline_routes.py --write")
    write_golden()
