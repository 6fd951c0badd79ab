"""ctypes binding of ``libkinectpy_b200.so`` (the C ABI declared in ``include/kp_api.h``).

This is the only door between the Python call surface and the CUDA kernels.  There is no CPU
implementation behind it: if the shared library has not been built, or no CUDA device is
visible, every operation raises ``KinectPyB200Error``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkinectpy_b200.so")

KP_OK, KP_E_ARG, KP_E_CUDA, KP_E_RANGE, KP_E_NOMEM, KP_E_NODEVICE = 0, -1, -2, -3, -4, -5
UNPROJECT_INT16 = 1
UNPROJECT_DROP_ANY_ZERO = 2
RESAMPLE_RANDOM, RESAMPLE_PREFIX = 0, 1
FLOOR_RANSAC, FLOOR_PLANE = 0, 1


class KinectPyB200Error(RuntimeError):
    """Raised for every failure of the native library (Open3D raises RuntimeError too)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"[kp {code}] {message}")
        self.code = code


class PipelineCfg(C.Structure):
    _fields_ = [
        ("S", C.c_int32), ("P", C.c_int64), ("unproject_flags", C.c_int32), ("scale", C.c_double),
        ("voxel_size", C.c_double), ("sor_k", C.c_int32), ("sor_ratio", C.c_double),
        ("do_floor", C.c_int32), ("floor_band", C.c_double), ("ransac_thr", C.c_double),
        ("ransac_n", C.c_int32), ("ransac_iters", C.c_int32),
        ("floor_sor_k", C.c_int32), ("floor_sor_ratio", C.c_double),
        ("do_icp", C.c_int32), ("icp_voxel", C.c_double), ("icp_max_corr", C.c_double), ("icp_max_iter", C.c_int32),
        ("normals_max_nn", C.c_int32), ("normals_radius", C.c_double),
        ("seed", C.c_uint64), ("n_streams", C.c_int32),
        ("do_crop", C.c_int32), ("crop_gate", C.c_double), ("resample_n", C.c_int32), ("resample_mode", C.c_int32),
        ("ror_nb_points", C.c_int32), ("ror_radius", C.c_double),
        ("floor_mode", C.c_int32), ("floor_plane", C.c_double * 4),
    ]


class FrameResult(C.Structure):
    _fields_ = [
        ("n_fused", C.c_int64), ("n_voxel", C.c_int64), ("n_sor", C.c_int64), ("n_floor_inliers", C.c_int64),
        ("n_out", C.c_int64),
        ("icp_T", (C.c_double * 16) * 5), ("icp_fitness", C.c_double * 5), ("icp_rmse", C.c_double * 5),
        ("icp_iters", C.c_int32 * 5), ("status", C.c_int32),
        ("floor_plane", C.c_double * 4),
    ]


_vp, _i32, _i64, _f64, _u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_uint64
_pi64, _pf64, _pi32, _pf32 = C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_float)

# name -> (restype, argtypes): must list every KP_EXPORT symbol of include/kp_api.h
SIGNATURES = {
    "kp_version": (C.c_char_p, []),
    "kp_device_count": (C.c_int, []),
    "kp_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "kp_ctx_destroy": (C.c_int, [_vp]),
    "kp_last_error": (C.c_char_p, [_vp]),
    "kp_ctx_stream": (_vp, [_vp]),
    "kp_sync": (C.c_int, [_vp]),
    "kp_malloc": (C.c_int, [_vp, C.c_size_t, C.POINTER(_vp)]),
    "kp_free": (C.c_int, [_vp, _vp]),
    "kp_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(_vp)]),
    "kp_host_free": (C.c_int, [_vp]),
    "kp_memcpy_h2d": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "kp_memcpy_d2h": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "kp_memcpy_d2d": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "kp_memset": (C.c_int, [_vp, _vp, C.c_int, C.c_size_t]),
    "kp_timer_start": (C.c_int, [_vp]),
    "kp_timer_stop": (C.c_int, [_vp, _pf32]),
    "kp_launch_count": (_i64, [_vp]),
    "kp_flush_l2": (C.c_int, [_vp]),
    "kp_profile_enable": (C.c_int, [_vp, C.c_int]),
    "kp_profile_read": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_char_p), _pf64, _pi64, _pf64, C.POINTER(C.c_int)]),
    "kp_profile_reset": (C.c_int, [_vp]),
    "kp_unproject_transform": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _i64, C.c_int, _f64, _vp, _vp, _vp, _vp, _vp]),
    "kp_points_from_xyz16": (C.c_int, [_vp, _vp, _i64, _vp, C.c_int, _f64, _vp, _vp, _vp]),
    "kp_crop_mask": (C.c_int, [_vp, _vp, _vp, _i64, _f64, _vp, _pf64]),
    "kp_transform_points": (C.c_int, [_vp, _vp, _i64, _vp, C.c_int]),
    "kp_bounds": (C.c_int, [_vp, _vp, _i64, _pf32, _pi64]),
    "kp_compact": (C.c_int, [_vp, _i64, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _pi64]),
    "kp_voxel_downsample": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _f64, _vp, _vp, _vp, _vp, _vp, _pf64, _pi64]),
    "kp_knn": (C.c_int, [_vp, _vp, _i64, _vp, _i64, C.c_int, _f64, _f64, _vp, _vp, _vp]),
    "kp_sor_mask": (C.c_int, [_vp, _vp, _i64, C.c_int, _f64, _f64, _vp, _vp, _pf64, _pi64]),
    "kp_radius_mask": (C.c_int, [_vp, _vp, _i64, C.c_int, _f64, _vp, _vp, _pi64]),
    "kp_estimate_normals": (C.c_int, [_vp, _vp, _i64, _f64, C.c_int, _vp]),
    "kp_ransac_plane": (C.c_int, [_vp, _vp, _i64, _f64, C.c_int, C.c_int, _f64, _u64, _pf64, _vp, _pi64, _pi32, _vp]),
    "kp_plane_side_mask": (C.c_int, [_vp, _vp, _i64, _f64, _f64, _f64, _f64, _vp, _pi64]),
    "kp_band_mask": (C.c_int, [_vp, _vp, _i64, C.c_int, _f64, _vp, _pf64, _pi64]),
    "kp_icp_point_to_plane": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _i64, _f64, _vp, C.c_int, _f64, _f64, _vp, _pf64, _pf64,
                                        C.POINTER(C.c_int), _pi64]),
    "kp_icp_point_to_point": (C.c_int, [_vp, _vp, _i64, _vp, _i64, _f64, _vp, C.c_int, _f64, _f64, _vp, _pf64, _pf64,
                                        C.POINTER(C.c_int), _pi64]),
    "kp_icp_colored": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _f64, _f64, _vp, C.c_int, _f64, _f64, _vp, _pf64, _pf64,
                                 C.POINTER(C.c_int), _pi64]),
    "kp_color_gradient": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _f64, C.c_int, _vp]),
    "kp_fpfh": (C.c_int, [_vp, _vp, _vp, _i64, _f64, C.c_int, _vp]),
    "kp_feature_match": (C.c_int, [_vp, _vp, _i64, _vp, _i64, C.c_int, _vp, _vp]),
    "kp_ransac_correspondence": (C.c_int, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _f64, C.c_int, _f64, _f64, C.c_int, _f64, _u64,
                                           _pf64, _pf64, _pf64, _pi32, _pi64]),
    "kp_resample_fixed_n": (C.c_int, [_vp, _vp, _i64, _i64, C.c_int, _u64, _u64, _vp, _vp, _pi64]),
    "kp_resample_batch": (C.c_int, [_vp, _vp, _pi64, C.c_int, _i64, C.c_int, _u64, _u64, _vp, _pi64]),
    "kp_pipeline_create": (C.c_int, [C.c_int, C.POINTER(PipelineCfg), _vp, _vp, C.POINTER(_vp)]),
    "kp_pipeline_destroy": (C.c_int, [_vp]),
    "kp_pipeline_last_error": (C.c_char_p, [_vp]),
    "kp_pipeline_run": (C.c_int, [_vp, _vp, C.c_int, _i64, C.POINTER(FrameResult), _vp, _i64]),
    "kp_pipeline_launch_count": (_i64, [_vp]),
    "kp_pipeline_frames_in_flight": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "kp_pipeline_frame_counts": (C.c_int, [_vp, _pi64, C.c_int]),
    "kp_pipeline_profile": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(C.c_char_p), _pf64, _pi64, _pf64, C.POINTER(C.c_int)]),
    "kp_pipeline_run_host": (C.c_int, [_vp, _vp, _i64, C.POINTER(FrameResult), _vp, _i64]),
    "kp_pipeline_run_ex": (C.c_int, [_vp, _vp, _vp, C.c_int, _i64, _vp, C.POINTER(FrameResult), _vp, _i64, _vp]),
}

_lib = None
_lib_lock = threading.Lock()


def load_library():
    """Load the shared library and attach the prototypes.  Raises if it was never built."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise KinectPyB200Error(KP_E_NODEVICE, f"{LIB_PATH} not found: build it with `make lib` "
                                    "(or `python -c 'import __graft_entry__ as g; g.build()'`); there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def _check(rc: int, ctx_handle=None):
    if rc != KP_OK:
        msg = load_library().kp_last_error(ctx_handle)
        raise KinectPyB200Error(rc, msg.decode() if msg else "unknown error")


class Context:
    """One CUDA stream + workspace (``kp_ctx``).  Not thread-safe: one per host thread."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = _vp()
        _check(self.lib.kp_ctx_create(device, C.byref(h)))
        self.handle = h
        self.device = device

    def close(self):
        if getattr(self, "handle", None):
            self.lib.kp_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int):
        _check(rc, self.handle)

    def sync(self):
        self.check(self.lib.kp_sync(self.handle))

    @property
    def stream(self) -> int:
        return int(self.lib.kp_ctx_stream(self.handle) or 0)

    def launch_count(self) -> int:
        return int(self.lib.kp_launch_count(self.handle))

    # -- memory ----------------------------------------------------------
    def empty(self, shape, dtype) -> "DeviceArray":
        return DeviceArray(self, shape, dtype)

    def to_device(self, arr: np.ndarray, dtype=None) -> "DeviceArray":
        a = np.ascontiguousarray(arr, dtype=dtype)
        d = DeviceArray(self, a.shape, a.dtype)
        if a.nbytes:
            self.check(self.lib.kp_memcpy_h2d(self.handle, d.ptr, a.ctypes.data, a.nbytes))
            self.sync()   # `a` may be a temporary: do not let it die before the copy ran
        return d

    # -- timing / profiling ----------------------------------------------
    def timer_start(self):
        self.check(self.lib.kp_timer_start(self.handle))

    def timer_stop(self) -> float:
        ms = C.c_float()
        self.check(self.lib.kp_timer_stop(self.handle, C.byref(ms)))
        return float(ms.value)

    def flush_l2(self):
        self.check(self.lib.kp_flush_l2(self.handle))

    def profile(self, on: bool):
        self.check(self.lib.kp_profile_reset(self.handle))
        self.check(self.lib.kp_profile_enable(self.handle, 1 if on else 0))

    def profile_read(self):
        names = (C.c_char_p * 64)()
        ms = (C.c_double * 64)()
        calls = (C.c_int64 * 64)()
        by = (C.c_double * 64)()
        n = C.c_int()
        self.check(self.lib.kp_profile_read(self.handle, 64, names, ms, calls, by, C.byref(n)))
        return {names[i].decode(): {"ms": float(ms[i]), "calls": int(calls[i]), "bytes": float(by[i])} for i in range(n.value)}


class DeviceArray:
    """A caller-owned device buffer (cudaMallocAsync on the context's stream)."""

    def __init__(self, ctx: Context, shape, dtype):
        self.ctx = ctx
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = _vp()
        ctx.check(ctx.lib.kp_malloc(ctx.handle, max(self.nbytes, 16), C.byref(p)))
        self.ptr = p.value

    def __del__(self):
        try:
            if self.ptr and self.ctx.handle:
                self.ctx.lib.kp_free(self.ctx.handle, self.ptr)
        except Exception:
            pass
        self.ptr = None

    def __len__(self):
        return self.shape[0] if self.shape else 0

    def to_host(self, rows: Optional[int] = None) -> np.ndarray:
        shape = self.shape if rows is None else (int(rows),) + self.shape[1:]
        out = np.empty(shape, dtype=self.dtype)
        if out.nbytes:
            self.ctx.check(self.ctx.lib.kp_memcpy_d2h(self.ctx.handle, out.ctypes.data, self.ptr, out.nbytes))
        return out

    def copy(self, rows: Optional[int] = None) -> "DeviceArray":
        shape = self.shape if rows is None else (int(rows),) + self.shape[1:]
        d = DeviceArray(self.ctx, shape, self.dtype)
        if d.nbytes:
            self.ctx.check(self.ctx.lib.kp_memcpy_d2d(self.ctx.handle, d.ptr, self.ptr, d.nbytes))
        return d

    def fill_bytes(self, value: int):
        if self.nbytes:
            self.ctx.check(self.ctx.lib.kp_memset(self.ctx.handle, self.ptr, value, self.nbytes))

    @property
    def __cuda_array_interface__(self):
        # lets torch.as_tensor(buf, device="cuda") view the buffer without a copy
        return {"shape": self.shape, "typestr": self.dtype.str, "data": (int(self.ptr or 0), False), "version": 3,
                "stream": self.ctx.stream or None}


def T16(T) -> np.ndarray:
    """4x4 (or None) -> contiguous float64[16], row-major."""
    a = np.ascontiguousarray(np.asarray(T, dtype=np.float64).reshape(4, 4))
    return a.reshape(16)


_default_ctx: dict = {}


def default_context(device: int = 0) -> Context:
    """Process-wide context per (thread, device); created on first use."""
    key = (threading.get_ident(), device)
    ctx = _default_ctx.get(key)
    if ctx is None or ctx.handle is None:
        ctx = Context(device)
        _default_ctx[key] = ctx
    return ctx


def device_available() -> bool:
    try:
        return load_library().kp_device_count() > 0
    except KinectPyB200Error:
        return False
