"""ctypes binding of libgsvc_rast.so (the C-ABI declared in include/gsvc_rast.h).

There is deliberately no fallback: if the library has not been built, or a symbol the header
declares is missing, loading raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgsvc_rast.so")
ABI_VERSION = 5

# gsvc_rast_status
OK, ERR_INVALID, ERR_CUDA, ERR_CAPACITY, ERR_OVERFLOW = 0, -1, -2, -3, -4


class Settings(C.Structure):
    """struct gsvc_rast_settings — the 13 fields of GaussianRasterizationSettings (renderer.py:63-83)."""
    _fields_ = [
        ("image_height", C.c_int32), ("image_width", C.c_int32),
        ("x_min", C.c_float), ("y_min", C.c_float), ("scale", C.c_float), ("threshold", C.c_float),
        ("bg", C.c_void_p), ("scale_modifier", C.c_float),
        ("viewmatrix", C.c_void_p), ("vm_stride_r", C.c_int64), ("vm_stride_c", C.c_int64),
        ("sh_degree", C.c_int32), ("campos", C.c_float * 3),
        ("prefiltered", C.c_int32), ("debug", C.c_int32),
    ]


class Exchange(C.Structure):
    """struct gsvc_rast_exchange — the rank-to-rank exchange a backward launch may carry."""
    _fields_ = [("multicast", C.c_void_p), ("buffers", C.c_void_p), ("signal_pads", C.c_void_p), ("state", C.c_void_p),
                ("rank", C.c_int32), ("world", C.c_int32), ("n_ctas", C.c_int32), ("chunk_rows", C.c_int32)]


EXCHANGE_MAX_CHUNKS = 62
EXCHANGE_STATE_WORDS = 2 + EXCHANGE_MAX_CHUNKS + 1     # go, done, chunk counters, count of waits that gave up


class View(C.Structure):
    """struct gsvc_rast_view — one view of a batched call (gsvc_rast_*_views)."""
    _fields_ = [
        ("viewmatrix", C.c_void_p), ("vm_stride_r", C.c_int64), ("vm_stride_c", C.c_int64),
        ("campos", C.c_float * 3), ("out_image", C.c_int32), ("flip_x", C.c_int32), ("weight", C.c_float),
    ]


MAX_VIEWS = 16

ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_int32, C.c_size_t)

_vp, _i32, _i64, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t
_SP = C.POINTER(Settings)
_VP = C.POINTER(View)

# name -> (restype, argtypes); must list every symbol include/gsvc_rast.h declares
SIGNATURES = {
    "gsvc_rast_abi_version": (C.c_int, []),
    "gsvc_rast_last_error": (C.c_char_p, []),
    "gsvc_rast_geom_bytes": (_sz, [_i32, _i32]),
    "gsvc_rast_image_bytes": (_sz, [_i32, _i32]),
    "gsvc_rast_image_bytes_views": (_sz, [_i32, _i32, _i32]),
    "gsvc_rast_binning_bytes": (_sz, [_i64]),
    "gsvc_rast_backward_scratch_bytes": (_sz, [_i32]),
    "gsvc_rast_visible_filter": (C.c_int, [_SP, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp]),
    "gsvc_rast_compact_scratch_bytes": (_sz, [_i32]),
    "gsvc_rast_visible_filter_compact": (C.c_int, [_SP, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_uint32,
                                                  _i32, _i32, _vp]),
    "gsvc_rast_forward_launch": (C.c_int, [_SP, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64,
                                           _vp, _vp, _vp, _vp, C.c_uint32, _vp]),
    "gsvc_rast_wait_count": (_i64, [_vp, C.c_uint32, _vp]),
    "gsvc_rast_forward_render": (C.c_int, [_SP, _i32, _vp, _vp, _vp, _i64, _vp, _vp]),
    "gsvc_rast_forward": (_i64, [_SP, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ALLOC_FN, _vp, _vp, _vp, _vp]),
    "gsvc_rast_backward": (C.c_int, [_SP, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                     _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gsvc_rast_forward_views_launch": (C.c_int, [_SP, _i32, _VP, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                                 _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, C.c_uint32, _vp]),
    "gsvc_rast_forward_views_render": (C.c_int, [_SP, _i32, _VP, _i32, _i32, _vp, _vp, _vp, _i64, _vp, _vp]),
    "gsvc_rast_backward_views": (C.c_int, [_SP, _i32, _VP, _i32, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                           _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                           _vp]),
    "gsvc_rast_backward_views_exchange": (C.c_int, [_SP, _i32, _VP, _i32, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                                    _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, C.POINTER(Exchange), _vp]),
    "gsvc_rast_forward_ragged_launch": (C.c_int, [_SP, _i32, _VP, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                                  _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, C.c_uint32, _vp]),
    "gsvc_rast_forward_ragged_render": (C.c_int, [_SP, _i32, _VP, _i32, _vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    "gsvc_rast_backward_ragged": (C.c_int, [_SP, _i32, _VP, _i32, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                            _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gsvc_rast_export_keys": (C.c_int, [_SP, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gsvc_rast_export_geom": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gsvc_rast_export_image": (C.c_int, [_SP, _i32, _vp, _vp, _vp, _vp]),
    "gsvc_rast_densify_stats": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _i64, _i32, _vp]),
    "gsvc_rast_switch_allreduce": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _i32, _vp]),
    "gsvc_rast_count_overflows": (C.c_int, [_i32]),
    "gsvc_rast_overflow_events": (_i64, [_i32, _vp]),
    "gsvc_rast_launch_count": (_i64, [_i32]),
    "gsvc_rast_stage_timing": (C.c_int, [_i32]),
    "gsvc_rast_stage_times": (C.c_int, [C.POINTER(C.c_float)]),
    "gsvc_gen_epilogue_scratch_bytes": (_sz, [_i32, _i32]),
    "gsvc_gen_epilogue_forward": (C.c_int, [_i32, _i32] + [_vp] * 20 + [_vp, C.c_uint32, _vp]),
    "gsvc_gen_epilogue_backward": (C.c_int, [_i32, _i32] + [_vp] * 26),
    "gsvc_rast_loss_scratch_bytes": (_sz, [_i32, _i32, _i32]),
    "gsvc_rast_loss_forward": (C.c_int, [_i32, _i32, _i32, _vp, _vp, C.c_float, _vp, _vp, _vp]),
    "gsvc_rast_loss_backward": (C.c_int, [_i32, _i32, _i32, _vp, _vp, C.c_float, _vp, _vp, _vp]),
    "gsvc_rast_quality_scratch_bytes": (_sz, [_i32, _i32, _i32]),
    "gsvc_rast_quality": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "gsvc_rast_frames_rgb8": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp]),
    "gsvc_rast_loss_forward_rgb8": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _i32, _vp, C.c_float, _vp, _vp, _vp]),
    "gsvc_rast_loss_backward_rgb8": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _i32, _vp, C.c_float, _vp, _vp, _vp]),
    "gsvc_rast_quality_rgb8": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
}

STAGES = ("preprocess", "tile_scan", "scatter", "sort_tiles", "render_forward", "render_backward",
          "preprocess_backward", "visible_filter")

_lib = None


class RasterizerError(RuntimeError):
    pass


def lib():
    """Load libgsvc_rast.so (once).  Raises if it is missing — there is no CPU or PyTorch fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RasterizerError(
            f"{LIB_PATH} is not built. Run `python -m gsvc_b200.build` (needs nvcc, targets sm_100a). "
            "gsvc_b200 has no CPU or PyTorch fallback for the rasterizer.")
    handle = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    got = handle.gsvc_rast_abi_version()
    if got != ABI_VERSION:
        raise RasterizerError(f"libgsvc_rast.so ABI version {got}, binding expects {ABI_VERSION}")
    _lib = handle
    return _lib


def check(rc: int, what: str):
    if rc < 0:
        msg = lib().gsvc_rast_last_error().decode("utf-8", "replace")
        raise RasterizerError(f"{what} failed (status {rc}): {msg}")
    return rc


def stage_timing(enable: bool):
    check(lib().gsvc_rast_stage_timing(1 if enable else 0), "gsvc_rast_stage_timing")


def stage_times() -> dict:
    """Milliseconds per stage for the most recent call (stages that did not run are omitted)."""
    buf = (C.c_float * len(STAGES))()
    check(lib().gsvc_rast_stage_times(buf), "gsvc_rast_stage_times")
    return {name: float(buf[i]) for i, name in enumerate(STAGES) if buf[i] >= 0}
