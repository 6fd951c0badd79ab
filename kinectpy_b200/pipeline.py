"""Batched whole-frame driver (BASELINE config C4) over ``kp_pipeline_*`` of the C ABI.

One ``FramePipeline`` = one GPU, driven by one host thread: frames go through the device in batches of B frames
per kernel launch with every intermediate count kept on the device (a CUDA graph per batch slot), so a call makes
no host round trip until its last batch is enqueued.  It replaces, for a stream of synchronised multi-sensor depth
frames, the per-frame body of ``DataProcessor.__init__`` (``preprocessing/data.py:35-69``: transform,
fuse, ``filter_outliers``) followed by the ``floor_removal.py:64-73`` loop body and a per-frame
``execute_point_to_plane_registration`` refinement of every sub sensor's extrinsic
(``preprocessing/registration.py:65-86``).  Frames are independent, so multi-GPU use is one
pipeline per rank over a disjoint slice of the frame indices (no collective on the frame path).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from . import _cabi
from ._cabi import FrameResult, KinectPyB200Error, PipelineCfg


@dataclass
class PipelineConfig:
    """Units follow ``scale`` (1e-3 -> metres, 1.0 -> millimetres); defaults are BASELINE's C4 in metres."""
    n_sensors: int = 3
    pixels: int = 1024 * 1024
    unproject_flags: int = _cabi.UNPROJECT_INT16 | _cabi.UNPROJECT_DROP_ANY_ZERO
    scale: float = 1e-3
    voxel_size: float = 0.01
    sor_k: int = 20
    sor_ratio: float = 2.0
    do_floor: bool = True
    floor_band: float = 0.20
    ransac_thr: float = 0.01
    ransac_n: int = 3
    ransac_iters: int = 1000
    floor_sor_k: int = 50
    floor_sor_ratio: float = 0.30
    do_icp: bool = True
    icp_voxel: float = 0.01
    icp_max_corr: float = 0.02
    icp_max_iter: int = 30
    normals_max_nn: int = 30
    normals_radius: float = 0.02
    seed: int = 1234
    n_streams: int = 4
    # human crop of the fused cloud (preprocessing/data.py:165-178): segmentation non-black and z <= median + gate (mm)
    do_crop: bool = False
    crop_gate: float = 750.0
    # fixed-N output per frame (the PointNet input): 0 = off, else N in 1..16384
    resample_n: int = 0
    resample_mode: int = _cabi.RESAMPLE_RANDOM
    # radius outlier removal after the SOR (remove_radius_outlier): 0 = off, else keep points with more than
    # ror_nb_points points (themselves included) closer than ror_radius (in the cloud's unit)
    ror_nb_points: int = 0
    ror_radius: float = 0.0

    def to_c(self) -> PipelineCfg:
        c = PipelineCfg()
        c.S, c.P, c.unproject_flags, c.scale = self.n_sensors, self.pixels, self.unproject_flags, self.scale
        c.voxel_size, c.sor_k, c.sor_ratio = self.voxel_size, self.sor_k, self.sor_ratio
        c.do_floor, c.floor_band, c.ransac_thr = int(self.do_floor), self.floor_band, self.ransac_thr
        c.ransac_n, c.ransac_iters = self.ransac_n, self.ransac_iters
        c.floor_sor_k, c.floor_sor_ratio = self.floor_sor_k, self.floor_sor_ratio
        c.do_icp, c.icp_voxel, c.icp_max_corr, c.icp_max_iter = int(self.do_icp), self.icp_voxel, self.icp_max_corr, self.icp_max_iter
        c.normals_max_nn, c.normals_radius = self.normals_max_nn, self.normals_radius
        c.seed, c.n_streams = self.seed, self.n_streams
        c.do_crop, c.crop_gate = int(self.do_crop), self.crop_gate
        c.resample_n, c.resample_mode = self.resample_n, self.resample_mode
        c.ror_nb_points, c.ror_radius = self.ror_nb_points, self.ror_radius
        return c


@dataclass
class FrameOutput:
    n_fused: int
    n_voxel: int
    n_sor: int
    n_floor_inliers: int
    n_out: int
    icp_T: np.ndarray          # [S-1,4,4] refined T_master<-sub
    icp_fitness: np.ndarray
    icp_rmse: np.ndarray
    icp_iters: np.ndarray
    points: Optional[np.ndarray] = None
    fixed: Optional[np.ndarray] = None     # [N,3] fixed-N slot (want_fixed); zeros for a frame with status != 0
    status: int = 0


class FramePipeline:
    def __init__(self, cfg: PipelineConfig, xy_tables: np.ndarray, T_fuse: np.ndarray, T_icp_init: Optional[np.ndarray] = None,
                 device: int = 0):
        self.lib = _cabi.load_library()
        self.cfg = cfg
        self.device = device
        S, P = cfg.n_sensors, cfg.pixels
        tab = np.ascontiguousarray(xy_tables, dtype=np.float32).reshape(S, P, 2)
        Tf = np.ascontiguousarray(T_fuse, dtype=np.float64).reshape(S, 16)
        Ti = Tf if T_icp_init is None else np.ascontiguousarray(T_icp_init, dtype=np.float64).reshape(S, 16)
        both = np.ascontiguousarray(np.stack([Tf, Ti]))
        h = C.c_void_p()
        c = cfg.to_c()
        rc = self.lib.kp_pipeline_create(device, C.byref(c), tab.ctypes.data, both.ctypes.data, C.byref(h))
        if rc != 0:
            raise KinectPyB200Error(rc, (self.lib.kp_last_error(None) or b"").decode())
        self.handle = h
        self._ctx = _cabi.default_context(device)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.kp_pipeline_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _raise(self, rc):
        raise KinectPyB200Error(rc, (self.lib.kp_pipeline_last_error(self.handle) or b"").decode())

    def upload(self, depth: np.ndarray, rgb: Optional[np.ndarray] = None):
        """depth uint16[F,S,P] -> device buffer for the HBM-resident leg; with ``rgb`` (uint8[F,S,P,3] segmentation
        images) -> (depth buffer, rgb buffer)."""
        d = self._ctx.to_device(depth, np.uint16)
        if rgb is None:
            self._ctx.sync()
            return d
        r = self._ctx.to_device(rgb, np.uint8)
        self._ctx.sync()
        return d, r

    def run(self, depth, rgb=None, n_frames: Optional[int] = None, want_points: bool = False, out_stride: Optional[int] = None,
            want_fixed: bool = False, frame_ids=None, check: bool = True):
        """depth: numpy uint16[F,S,P] (host: H2D inside the call) or a DeviceArray from ``upload``; rgb: the segmentation
        images uint8[F,S,P,3] in the same memory space (required exactly when the pipeline crops).  ``want_fixed``: each
        frame's fixed-N slot in ``FrameOutput.fixed`` (needs ``resample_n``); ``frame_ids`` int64[F] (default 0..F-1):
        its sample stream.  ``check=False`` returns the outputs of a call whose frames carry a status instead of raising
        (``FrameOutput.status``)."""
        S, P = self.cfg.n_sensors, self.cfg.pixels
        on_dev = isinstance(depth, _cabi.DeviceArray)
        if on_dev:
            F = int(depth.shape[0]) if n_frames is None else int(n_frames)
            ptr = depth.ptr
            rptr = rgb.ptr if rgb is not None else None
        else:
            depth = np.ascontiguousarray(depth, dtype=np.uint16).reshape(-1, S, P)
            F = depth.shape[0] if n_frames is None else int(n_frames)
            ptr = depth.ctypes.data
            if rgb is not None:
                rgb = np.ascontiguousarray(rgb, dtype=np.uint8).reshape(-1, S, P, 3)
            rptr = rgb.ctypes.data if rgb is not None else None
        res = (FrameResult * F)()
        out = None
        stride = 0
        if want_points:
            stride = int(out_stride or S * P)
            out = self._ctx.empty((F, stride, 3), np.float32)
            self._ctx.sync()
        fixed = None
        if want_fixed:
            fixed = self._ctx.empty((F, max(int(self.cfg.resample_n), 1), 3), np.float32)
            self._ctx.sync()
        ids = None
        if frame_ids is not None:
            ids = np.ascontiguousarray(frame_ids, dtype=np.int64).reshape(-1)
            if ids.size != F:
                raise ValueError("frame_ids must hold one id per frame")
        rc = self.lib.kp_pipeline_run_ex(self.handle, ptr, rptr, 1 if on_dev else 0, F, ids.ctypes.data if ids is not None else None,
                                         res, out.ptr if out is not None else None, stride, fixed.ptr if fixed is not None else None)
        if rc != 0 and (check or all(res[f].status == 0 for f in range(F))):      # (a call-level error has no frame status)
            self._raise(rc)
        outs: List[FrameOutput] = []
        host = out.to_host() if out is not None else None
        hfixed = fixed.to_host() if fixed is not None else None
        for f in range(F):
            r = res[f]
            T = np.array([list(r.icp_T[i]) for i in range(max(S - 1, 0))], dtype=np.float64).reshape(-1, 4, 4)
            fo = FrameOutput(r.n_fused, r.n_voxel, r.n_sor, r.n_floor_inliers, r.n_out, T,
                             np.array(list(r.icp_fitness)[:S - 1]), np.array(list(r.icp_rmse)[:S - 1]),
                             np.array(list(r.icp_iters)[:S - 1]))
            fo.status = int(r.status)
            if host is not None:
                fo.points = host[f, :r.n_out].copy()
            if hfixed is not None:
                fo.fixed = hfixed[f].copy()
            outs.append(fo)
        self._last_raw = res
        return outs

    def run_raw(self, depth_ptr: int, on_device: bool, n_frames: int, d_out_ptr=None, out_stride: int = 0):
        """Timing form: no numpy conversion of the results (returns the ctypes result array).  ``d_out_ptr``:
        optional device buffer ``float32 [n_frames][out_stride][3]`` receiving each frame's final cloud."""
        res = (FrameResult * n_frames)()
        rc = self.lib.kp_pipeline_run(self.handle, depth_ptr, 1 if on_device else 0, n_frames, res, d_out_ptr, out_stride)
        if rc != 0:
            self._raise(rc)
        return res

    def run_host(self, h_depth_ptr: int, n_frames: int, h_out_ptr: int, out_stride: int):
        """End-to-end form: host depth in, results struct + each frame's final cloud out to host memory."""
        res = (FrameResult * n_frames)()
        rc = self.lib.kp_pipeline_run_host(self.handle, h_depth_ptr, n_frames, res, h_out_ptr, out_stride)
        if rc != 0:
            self._raise(rc)
        return res

    def frames_in_flight(self):
        """(frames per kernel launch, batch slots in flight) the pipeline was built with."""
        b, w = C.c_int(), C.c_int()
        self.lib.kp_pipeline_frames_in_flight(self.handle, C.byref(b), C.byref(w))
        return b.value, w.value

    def frame_counts(self) -> dict:
        """Device-side counts of the first frame of the last batch on slot 0 (diagnostics, byte accounting)."""
        v = (C.c_int64 * 36)()
        rc = self.lib.kp_pipeline_frame_counts(self.handle, v, 36)
        if rc != 0:
            self._raise(rc)
        S = self.cfg.n_sensors
        d = dict(zip(("n_fused", "n_voxel", "n_sor", "n_lo", "n_rest", "n_merged", "n_fsor", "n_out"), [int(x) for x in v[:8]]))
        d["n_inl"] = d["n_lo"] - d["n_rest"]
        d["leftovers_l0"], d["leftovers_l1"] = [int(x) for x in v[8:11]], [int(x) for x in v[11:14]]
        d["leftovers_mid"] = [int(x) for x in v[26:29]]      # (the ICP target's search has no mid level: [2] is 0)
        d["nv_icp"], d["n_icp"] = [int(x) for x in v[14:14 + S]], [int(x) for x in v[20:20 + S]]
        d["crop_median"] = [int(x) / 2.0 for x in v[29:29 + S]]     # (0.0 without the crop)
        d["n_ror"] = int(v[35])                                      # (0 without the radius outlier removal)
        return d

    def launch_count(self) -> int:
        return int(self.lib.kp_pipeline_launch_count(self.handle))

    def profile(self, on: bool):
        rc = self.lib.kp_pipeline_profile(self.handle, 1 if on else 0, 0, None, None, None, None, None)
        if rc != 0:
            self._raise(rc)

    def profile_read(self):
        names = (C.c_char_p * 64)()
        ms = (C.c_double * 64)()
        calls = (C.c_int64 * 64)()
        by = (C.c_double * 64)()
        n = C.c_int()
        rc = self.lib.kp_pipeline_profile(self.handle, 2, 64, names, ms, calls, by, C.byref(n))
        if rc != 0:
            self._raise(rc)
        return {names[i].decode(): {"ms": float(ms[i]), "calls": int(calls[i]), "bytes": float(by[i])} for i in range(n.value)}
