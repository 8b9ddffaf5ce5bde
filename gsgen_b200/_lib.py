"""ctypes binding of libgsb200.so (C ABI: include/gsb200.h).

There is deliberately no fallback: if the shared library is missing or a tensor is not a CUDA
tensor the call raises.  `python -m gsgen_b200.build` (or `__graft_entry__.build()`) compiles it.
"""
from __future__ import annotations

import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GSB200_LIB", os.path.join(_HERE, "libgsb200.so"))  # env override: tuning builds only

c_void = ctypes.c_void_p
c_u32 = ctypes.c_uint32
c_i32 = ctypes.c_int32
c_f32 = ctypes.c_float
c_i64 = ctypes.c_int64

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED, ERR_MISMATCH, ERR_OVERFLOW = 0, 1, 2, 3, 4, 5
OPT_BWD_SH_VARIANT, OPT_ASYNC_COUNT = 1, 2  # GSB200_OPT_* (include/gsb200.h)


class Gsb200Camera(ctypes.Structure):
    _fields_ = [
        ("c2w", c_f32 * 12),
        ("fx", c_f32), ("fy", c_f32), ("cx", c_f32), ("cy", c_f32),
        ("W", c_i32), ("H", c_i32),
        ("frustum_normals", c_f32 * 18),
        ("frustum_pts", c_f32 * 18),
        ("frustum_radius", c_f32),
        ("tile_radius", c_f32),
        ("T_thresh", c_f32),
        ("skip_frustum_culling", c_i32),
        ("depth_detach", c_i32),
    ]


class Gsb200ViewIn(ctypes.Structure):
    _fields_ = [
        ("N", c_u32),
        ("mean", c_void), ("qvec", c_void), ("svec", c_void), ("alpha", c_void),
        ("color", c_void), ("sh", c_void),
        ("C", c_i32),
        ("sh_c2w9", c_f32 * 9),
        ("bg", c_void), ("bg_rgb", c_void),
        ("act", c_i32),
    ]


class Gsb200AdamField(ctypes.Structure):
    _fields_ = [("begin", ctypes.c_uint64), ("count", ctypes.c_uint64), ("lr", ctypes.c_double)]


ACT_SVEC_EXP, ACT_ALPHA_SIGMOID, ACT_COLOR_SIGMOID = 1, 2, 4  # GSB200_ACT_* (include/gsb200.h)


class Gsb200ViewOut(ctypes.Structure):
    _fields_ = [
        ("rgb", c_void), ("T", c_void), ("depth", c_void), ("opacity", c_void), ("z2", c_void),
        ("mean2d", c_void), ("cov2d", c_void), ("depthg", c_void), ("mask", c_void), ("radii2d", c_void),
        ("h_num_dup", ctypes.POINTER(c_i64)),
        ("h_generation", ctypes.POINTER(c_i64)),
    ]


class Gsb200ViewGrads(ctypes.Structure):
    _fields_ = [
        ("g_rgb", c_void), ("rgb", c_void),
        ("g_depth", c_void), ("depth", c_void),
        ("g_opacity", c_void), ("opacity", c_void),
        ("g_z2", c_void), ("z2", c_void),
        ("T", c_void),
        ("mask", c_void),
        ("g_mean", c_void), ("g_qvec", c_void), ("g_svec", c_void), ("g_alpha", c_void),
        ("g_color", c_void), ("g_sh", c_void), ("g_mean2d", c_void), ("g_bg", c_void),
        ("accumulate", c_i32),
        ("generation", c_i64),
        ("touched", c_void),
    ]


_lib = None
_lock = threading.Lock()
_ctxs = {}  # (device index, slot) -> gsb200_ctx*

# every symbol include/gsb200.h declares (checked by the CPU test-suite)
EXPORTS = [
    "gsb200_last_error", "gsb200_version", "gsb200_ctx_create", "gsb200_ctx_destroy",
    "gsb200_culling_gaussian_bsphere", "gsb200_tile_culling_aabb_start_end",
    "gsb200_tile_based_vol_rendering_start_end_with_T", "gsb200_tile_based_vol_rendering_backward_start_end",
    "gsb200_tile_based_vol_rendering_scalar", "gsb200_tile_based_vol_rendering_scalar_backward",
    "gsb200_tile_based_vol_rendering_sh", "gsb200_tile_based_vol_rendering_backward_sh",
    "gsb200_project_gaussians_forward", "gsb200_project_gaussians_backward", "gsb200_tile_culling_aabb_count",
    "gsb200_render_forward", "gsb200_render_backward", "gsb200_view_stats",
    "gsb200_ctx_set_profiling", "gsb200_ctx_get_profile", "gsb200_adam_step", "gsb200_ctx_set_option",
    "gsb200_store_compact", "gsb200_store_append", "gsb200_rows_pack", "gsb200_rows_unpack", "gsb200_knn",
    "gsb200_estimate_normals", "gsb200_estimate_normals_backward",
]


def lib():
    """Load libgsb200.so (once).  Raises if it has not been built -- no fallback."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} not found: build the CUDA library first (python -m gsgen_b200.build). "
                        "gsgen_b200 has no CPU or PyTorch fallback.")
                L = ctypes.CDLL(LIB_PATH)
                L.gsb200_last_error.restype = ctypes.c_char_p
                for name in EXPORTS[1:]:
                    getattr(L, name).restype = ctypes.c_int
                _lib = L
    return _lib


class TileListOverflow(RuntimeError):
    """asynchronous-count mode: the view did not fit the tile-list capacity; render it again"""


def check(rc: int):
    if rc != OK:
        msg = lib().gsb200_last_error().decode("utf-8", "replace")
        raise (TileListOverflow if rc == ERR_OVERFLOW else RuntimeError)(f"libgsb200 error {rc}: {msg}")


def set_option(device: torch.device, slot: int, option: int, value: int):
    check(lib().gsb200_ctx_set_option(ctx(device, slot), ctypes.c_int(option), ctypes.c_int64(value)))


def ctx(device: torch.device, slot: int = 0):
    """Per-(device, slot) context: scratch arena + saved state of one in-flight view."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    key = (idx, slot)
    c = _ctxs.get(key)
    if c is None:
        p = ctypes.c_void_p()
        check(lib().gsb200_ctx_create(int(idx), ctypes.byref(p)))
        _ctxs[key] = c = p
    return c


def stream_ptr(device: torch.device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t, dtype=None, name="tensor"):
    """data_ptr of a contiguous CUDA tensor with the reference's contract (CHECK_DC_*, common.h:46-54)."""
    if t is None:
        return ctypes.c_void_p(0)
    if not isinstance(t, torch.Tensor):
        raise RuntimeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be a contiguous tensor")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"{name} must be a {dtype} tensor, got {t.dtype}")
    return ctypes.c_void_p(t.data_ptr())


def fptr(t, name="tensor"):
    return ptr(t, torch.float32, name)


def iptr(t, name="tensor"):
    return ptr(t, torch.int32, name)
