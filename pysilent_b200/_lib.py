"""ctypes binding of ``libsilent_b200.so`` (C ABI declared in ``include/silent_b200.h``).

There is NO CPU fallback: if the library has not been built (``python -m pysilent_b200.build`` or
``__graft_entry__.build()``) every operator raises ``RuntimeError``. ctypes releases the GIL for the duration of each
call, so the pipeline can be driven from one Python thread per camera like the reference's cvpubsubs callback threads.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsilent_b200.so")

SILENT_U8, SILENT_F32, SILENT_NV12 = 0, 1, 2
POST_NONE, POST_RELU, POST_RELU_CLIP = 0, 1, 2
PW_DIV255, PW_INVERT255, PW_IMPORTANCE, PW_MUL255, PW_ENERGY_DISPLAY, PW_PRODUCT = range(6)

# every symbol include/silent_b200.h declares (tests check the .so exports exactly these)
SYMBOLS = (
    "silent_abi_version", "silent_last_error", "silent_launch_count", "silent_device_count",
    "silent_plan_enable_timing", "silent_plan_stage_ms", "silent_plan_stack_split_ms", "silent_plan_create", "silent_plan_destroy",
    "silent_plan_reserve", "silent_plan_levels", "silent_plan_level_hw", "silent_plan_level_info",
    "silent_plan_level_tables", "silent_plan_algorithmic_bytes", "silent_pyramid_build", "silent_conv2d",
    "silent_regulate", "silent_pad_inwards", "silent_value_from_color", "silent_selection_workspace_bytes",
    "silent_max_value_indices_region", "silent_top_value_points", "silent_stack_workspace_bytes", "silent_stack_fused", "silent_pipeline_run",
    "silent_pipeline_run_host", "silent_pipeline_run_bank", "silent_pipeline_run_orientations", "silent_stack_bank", "silent_get_centroids", "silent_resize_nearest", "silent_get_boosting", "silent_pointwise", "silent_display_tensors",
    "silent_display_sequence_scratch_bytes", "silent_display_sequence", "silent_pack_points",
    "silent_comm_unique_id", "silent_comm_create", "silent_comm_destroy", "silent_comm_check", "silent_gather_points",
    "silent_stack_fused_f16", "silent_stack_bank_f16", "silent_pipeline_run_f16", "silent_pipeline_run_orientations_f16",
    "silent_pipeline_run_host_f16", "silent_nv12_to_bgr", "silent_plan_level_coords", "silent_point_records",
    "silent_point_patches", "silent_peak_points", "silent_plan_peak_points", "silent_match_points",
    "silent_motion_workspace_bytes", "silent_estimate_motion",
)


class SilentParams(ctypes.Structure):
    _fields_ = [("frame_h", ctypes.c_int32), ("frame_w", ctypes.c_int32), ("frame_c", ctypes.c_int32),
                ("num_colors", ctypes.c_int32), ("center_w", ctypes.c_int32), ("center_h", ctypes.c_int32),
                ("scale", ctypes.c_double), ("frame_dtype", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class SilentStackWeights(ctypes.Structure):
    _fields_ = [("rgc", ctypes.c_float * 81), ("rgby", ctypes.c_float * 81), ("stripe", ctypes.c_float * 81),
                ("blur", ctypes.c_float * 441), ("end", ctypes.c_float * 81), ("regulation_value", ctypes.c_float),
                ("regulation_root", ctypes.c_float), ("clip_max", ctypes.c_float), ("border", ctypes.c_int32)]


class SilentBankWeights(ctypes.Structure):
    """silent_bank_weights: the 8-orientation bank of BASELINE config C4."""
    _fields_ = [("rgc", ctypes.c_float * 81), ("rgby", ctypes.c_float * 81), ("stripe", ctypes.c_float * (9 * 3 * 8)),
                ("blur", ctypes.c_float * (49 * 64)), ("end", ctypes.c_float * (9 * 64)),
                ("regulation_value", ctypes.c_float), ("regulation_root", ctypes.c_float), ("clip_max", ctypes.c_float),
                ("border", ctypes.c_int32)]


BANK_MAX = 16                  # SILENT_BANK_MAX
FUSED_BANK_WIDTHS = (4, 8, 12, 16)   # orientation counts with fused kernels (silent_pipeline_run_orientations)
RECORD_CHANNELS = (3,) + FUSED_BANK_WIDTHS   # output channel counts silent_point_records reads
PATCH_RADIUS_MAX = 31          # SILENT_PATCH_RADIUS_MAX: largest radius silent_point_patches takes
MOTION_HYPOTHESES_MAX = 4096   # SILENT_MOTION_HYPOTHESES_MAX: most hypotheses silent_estimate_motion takes


class SilentOrientationBank(ctypes.Structure):
    """silent_orientation_bank: a bank of ``orientations`` = 4, 8, 12 or 16; each filter packed densely at the front of
    an array sized for ``BANK_MAX``."""
    _fields_ = [("orientations", ctypes.c_int32), ("rgc", ctypes.c_float * 81), ("rgby", ctypes.c_float * 81),
                ("stripe", ctypes.c_float * (9 * 3 * BANK_MAX)), ("blur", ctypes.c_float * (49 * BANK_MAX * BANK_MAX)),
                ("end", ctypes.c_float * (9 * BANK_MAX * BANK_MAX)), ("regulation_value", ctypes.c_float),
                ("regulation_root", ctypes.c_float), ("clip_max", ctypes.c_float), ("border", ctypes.c_int32)]


_lib = None


def lib():
    """Load the shared library once; fail loudly if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "pysilent_b200: %s is missing. Build it with `python -m pysilent_b200.build` (needs nvcc); "
            "there is no CPU fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    i, f, d, p, sz, i64 = ctypes.c_int, ctypes.c_float, ctypes.c_double, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int64
    ip = ctypes.POINTER(ctypes.c_int)
    sig = {
        "silent_abi_version": (i, []),
        "silent_last_error": (ctypes.c_char_p, []),
        "silent_device_count": (i, []),
        "silent_launch_count": (i64, []),
        "silent_plan_enable_timing": (i, [p, i]),
        "silent_plan_stage_ms": (i, [p, ctypes.POINTER(f), ctypes.POINTER(f), ctypes.POINTER(f)]),
        "silent_plan_stack_split_ms": (i, [p, ctypes.POINTER(f), ctypes.POINTER(f)]),
        "silent_plan_create": (i, [ctypes.POINTER(SilentParams), ctypes.POINTER(p)]),
        "silent_plan_destroy": (None, [p]),
        "silent_plan_reserve": (i, [p, i]),
        "silent_plan_levels": (i, [p]),
        "silent_plan_level_hw": (i, [p, ip, ip]),
        "silent_plan_level_info": (i, [p, i, ip, ip, ip, ip, ip, ip]),
        "silent_plan_level_tables": (i, [p, i, p, p, p, p]),
        "silent_plan_level_coords": (i, [p, i, p, p]),
        "silent_plan_algorithmic_bytes": (i64, [p]),
        "silent_pyramid_build": (i, [p, p, i, p, p]),
        "silent_conv2d": (i, [p, i, i, i, i, p, i, i, i, f, p, p]),
        "silent_regulate": (i, [p, i, i, i, i, p, i, f, f, p, p]),
        "silent_pad_inwards": (i, [p, i, i, i, i, i, i, i, i, p, p]),
        "silent_value_from_color": (i, [p, i, i, i, i, p, p]),
        "silent_selection_workspace_bytes": (sz, [i, i, i]),
        "silent_max_value_indices_region": (i, [p, i, i, i, i, i, p, i64, p, p, sz, p]),
        "silent_top_value_points": (i, [p, p, i, i, i, i, d, p, p, sz, p]),
        "silent_peak_points": (i, [p, i, i, i, d, p, i64, p, p, sz, p]),
        "silent_plan_peak_points": (i, [p, i, d, p, i64, p, p]),
        "silent_stack_workspace_bytes": (sz, [i, i, i]),
        "silent_stack_fused": (i, [p, i, i, i, ctypes.POINTER(SilentStackWeights), p, p, p, p, sz, p]),
        "silent_pipeline_run": (i, [p, ctypes.POINTER(SilentStackWeights), p, i, p, p, p, p, i64, p, p]),
        "silent_pipeline_run_host": (i, [p, ctypes.POINTER(SilentStackWeights), p, i, p, p, p, i64, p, p]),
        "silent_pipeline_run_bank": (i, [p, ctypes.POINTER(SilentBankWeights), p, i, p, p, p, i64, p, p]),
        "silent_pipeline_run_orientations": (i, [p, ctypes.POINTER(SilentOrientationBank), p, i, p, p, p, i64, p, p]),
        "silent_stack_bank": (i, [p, i, i, i, ctypes.POINTER(SilentOrientationBank), p, p, p, p, sz, p]),
        # binary16 outputs: the same arguments, orient / line_end as uint16_t bit patterns (np.float16, torch.float16)
        "silent_stack_fused_f16": (i, [p, i, i, i, ctypes.POINTER(SilentStackWeights), p, p, p, p, sz, p]),
        "silent_stack_bank_f16": (i, [p, i, i, i, ctypes.POINTER(SilentOrientationBank), p, p, p, p, sz, p]),
        "silent_pipeline_run_f16": (i, [p, ctypes.POINTER(SilentStackWeights), p, i, p, p, p, p, i64, p, p]),
        "silent_pipeline_run_orientations_f16": (i, [p, ctypes.POINTER(SilentOrientationBank), p, i, p, p, p, i64, p, p]),
        "silent_pipeline_run_host_f16": (i, [p, ctypes.POINTER(SilentStackWeights), p, i, p, p, p, i64, p, p]),
        "silent_nv12_to_bgr": (i, [p, i, i, i, p, p]),
        "silent_point_records": (i, [p, i, p, p, i64, p, p, i, i, p, p, p, p, p]),
        "silent_point_patches": (i, [p, i, p, p, i64, p, p, i, i, p, i, p, p, p, p]),
        "silent_match_points": (i, [p, p, i64, p, i64, i, i, f, p, p, p, p]),
        "silent_motion_workspace_bytes": (sz, [i64]),
        "silent_estimate_motion": (i, [p, p, p, p, i64, i, i, f, ctypes.c_uint64, p, sz, p, p, p, p, p]),
        "silent_get_centroids": (i, [p, i, i, i, i, i, p, p, p, p]),
        "silent_resize_nearest": (i, [p, i, i, i, i, i, i, p, p]),
        "silent_get_boosting": (i, [p, p, i, i, i, f, f, i, p, p, p]),
        "silent_pointwise": (i, [p, p, sz, i, p, p]),
        "silent_display_tensors": (i, [p, i, i, i, i, i, i, i, p, f, f, i, f, f, p, p, p, p, p, p]),
        "silent_display_sequence_scratch_bytes": (sz, [i, i, i, i, i, i]),
        "silent_display_sequence": (i, [p, i, i, i, i, i, i, i, i, p, f, f, i, f, f, p, p, p, p, p, sz, p]),
        "silent_pack_points": (i, [p, p, i64, i64, p, p]),
        "silent_comm_unique_id": (i, [p]),
        "silent_comm_create": (i, [p, i, i, ctypes.POINTER(p)]),
        "silent_comm_destroy": (None, [p]),
        "silent_comm_check": (i, [p]),
        "silent_gather_points": (i, [p, p, i64, p, p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    if L.silent_abi_version() != 1:
        raise RuntimeError("pysilent_b200: ABI version mismatch in %s" % LIB_PATH)
    _lib = L
    return L


def check(rc, what=""):
    """Map a negative silent_status to RuntimeError (SURVEY 8(b): C-ABI codes surface as RuntimeError)."""
    if rc is not None and rc < 0:
        msg = lib().silent_last_error().decode("utf-8", "replace")
        raise RuntimeError("libsilent_b200 %s failed (status %d): %s" % (what, rc, msg))
    return rc


def _pack(w, who, filters, regulation_value, regulation_root, clip_max, border):
    """Copy ``(name, array, shape)`` HWIO filters into the struct ``w``, rounded to float32 like ``tf.constant(...,
    tf.float32)``; a filter of another shape raises ValueError ("<who> needs <name> of shape ...")."""
    for name, arr, shape in filters:
        a = np.ascontiguousarray(np.asarray(arr), dtype=np.float32)
        if a.shape != shape:
            raise ValueError("%s needs %s of shape %s, got %s" % (who, name, shape, a.shape))
        ctypes.memmove(getattr(w, name), a.ctypes.data, a.nbytes)
    w.regulation_value, w.regulation_root, w.clip_max, w.border = regulation_value, regulation_root, clip_max, border
    return w


def make_stack_weights(rgc, rgby, stripe, blur, end, regulation_value=1.0, regulation_root=.1, clip_max=255.0, border=2):
    """Pack HWIO filters (any float dtype) into the C struct, rounding to float32 like ``tf.constant(..., tf.float32)``."""
    return _pack(SilentStackWeights(), "fused stack",
                 (("rgc", rgc, (3, 3, 3, 3)), ("rgby", rgby, (3, 3, 3, 3)), ("stripe", stripe, (3, 3, 3, 3)),
                  ("blur", blur, (7, 7, 3, 3)), ("end", end, (3, 3, 3, 3))),
                 regulation_value, regulation_root, clip_max, border)


def make_bank_weights(rgc, rgby, stripe, blur, end, regulation_value=1.0, regulation_root=.1, clip_max=255.0, border=2):
    """Pack the 8-orientation bank (HWIO, any float dtype) into ``silent_bank_weights``."""
    return _pack(SilentBankWeights(), "the fused orientation bank",
                 (("rgc", rgc, (3, 3, 3, 3)), ("rgby", rgby, (3, 3, 3, 3)), ("stripe", stripe, (3, 3, 3, 8)),
                  ("blur", blur, (7, 7, 8, 8)), ("end", end, (3, 3, 8, 8))),
                 regulation_value, regulation_root, clip_max, border)


def make_orientation_bank(rgc, rgby, stripe, blur, end, regulation_value=1.0, regulation_root=.1, clip_max=255.0,
                          border=2):
    """Pack an orientation bank (HWIO, any float dtype) into ``silent_orientation_bank``. The width n is the stripe
    bank's output count; blur must be [7,7,n,n] and end [3,3,n,n]. Whether the library has fused kernels for n (4, 8, 12,
    16) is checked by the library itself."""
    st = np.asarray(stripe).shape
    if len(st) != 4 or st[:3] != (3, 3, 3) or not 1 <= st[3] <= BANK_MAX:
        raise ValueError("an orientation bank needs a stripe bank of shape (3, 3, 3, n) with 1 <= n <= %d, got %s"
                         % (BANK_MAX, st))
    n = st[3]
    w = SilentOrientationBank()
    w.orientations = n
    return _pack(w, "a %d-orientation bank" % n,
                 (("rgc", rgc, (3, 3, 3, 3)), ("rgby", rgby, (3, 3, 3, 3)), ("stripe", stripe, (3, 3, 3, n)),
                  ("blur", blur, (7, 7, n, n)), ("end", end, (3, 3, n, n))),
                 regulation_value, regulation_root, clip_max, border)
