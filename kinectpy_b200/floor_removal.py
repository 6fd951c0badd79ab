"""B200 counterpart of the reference's ``floor_removal.py``.

``equation_plane`` and ``pcd_above_plane`` keep their signatures (``floor_removal.py:21,39``); the
per-point Python loop of ``pcd_above_plane`` (``floor_removal.py:42-48``) becomes one mask kernel
plus an ordered compaction.  ``remove_floor`` is the body of the script's loop
(``floor_removal.py:64-73``) as a function: floor band by max-y, RANSAC plane on the band, keep the
band's non-plane points, merge with the upper part, statistical outlier removal.  ``remove_floor_batch``
runs that body over a list of clouds in one batched frame-engine pipeline.
"""
from __future__ import annotations

import ctypes as C
import glob
import os

import numpy as np

from . import _cabi, geometry
from .geometry import PointCloud
from .io_formats import read_point_cloud, write_point_cloud


def pick_points(pcd):
    raise NotImplementedError("interactive point picking needs the Open3D GUI (out of scope, SURVEY.md section 2 row 7)")


def equation_plane(p1, p2, p3):
    """Plane through three points: unnormalised cross-product normal, ``d = -n.p1`` (``floor_removal.py:21-36``)."""
    p1, p2, p3 = (np.asarray(p, dtype=np.float64) for p in (p1, p2, p3))
    u, v = p2 - p1, p3 - p1
    a = u[1] * v[2] - v[1] * u[2]
    b = v[0] * u[2] - u[0] * v[2]
    c = u[0] * v[1] - u[1] * v[0]
    d = -a * p1[0] - b * p1[1] - c * p1[2]
    print("equation of plane is ", a, "x +", b, "y +", c, "z +", d, "= 0.")
    return a, b, c, d


def pcd_above_plane(a, b, c, d, pcd: PointCloud) -> PointCloud:
    """Keep the points with ``a*x + b*y + c*z + d < 0`` (``floor_removal.py:39-51``)."""
    n = len(pcd)
    if n == 0:
        return PointCloud()
    ctx, pts, _, _ = pcd._dev()
    mask = ctx.empty((n,), np.uint8)
    kept = C.c_int64()
    ctx.check(ctx.lib.kp_plane_side_mask(ctx.handle, pts.ptr, n, float(a), float(b), float(c), float(d), mask.ptr,
                                         C.byref(kept)))
    out, _ = pcd._select_mask(mask, want_index=False)
    return out


def split_floor_band(pcd: PointCloud, band: float = 200, axis: int = 1):
    """(lower, upper): lower = points with ``coord >= max(coord) - band`` (``floor_removal.py:64-69``)."""
    n = len(pcd)
    if n == 0:
        return PointCloud(), PointCloud()
    ctx, pts, _, _ = pcd._dev()
    mask = ctx.empty((n,), np.uint8)
    nlow = C.c_int64()
    amax = C.c_double()
    ctx.check(ctx.lib.kp_band_mask(ctx.handle, pts.ptr, n, int(axis), float(band), mask.ptr, C.byref(amax), C.byref(nlow)))
    lower, _ = pcd._select_mask(mask, invert=False, want_index=False)
    upper, _ = pcd._select_mask(mask, invert=True, want_index=False)
    return lower, upper


def remove_floor(pcd: PointCloud, band: float = 200, distance_threshold: float = 30, ransac_n: int = 30,
                 num_iterations: int = 2000, nb_neighbors: int = 50, std_ratio: float = 0.30, seed=None,
                 return_details: bool = False):
    """One iteration of the reference script's loop body (``floor_removal.py:64-73``), same literals as defaults."""
    floor, upper = split_floor_band(pcd, band)
    plane_model, inliers = floor.segment_plane(distance_threshold=distance_threshold, ransac_n=ransac_n,
                                               num_iterations=num_iterations, seed=seed)
    outlier_cloud = floor.select_by_index(inliers, invert=True)   # feet and whatever else is not floor
    merged = outlier_cloud + upper
    filtered, _ = merged.remove_statistical_outlier(nb_neighbors, std_ratio)
    if return_details:
        return filtered, plane_model, inliers
    return filtered


def remove_floor_batch(pcds, band: float = 200, distance_threshold: float = 30, ransac_n: int = 30, num_iterations: int = 2000,
                       nb_neighbors: int = 50, std_ratio: float = 0.30, seed=None, spacing: float = 10.0, n_streams: int = 16):
    """``remove_floor`` over a list of clouds in one batched frame-engine pipeline (cloud input, no voxel step): the same
    literals, the same results, without a host round trip per cloud.  ``spacing``: the clouds' typical point spacing in
    their unit (millimetres for the literals above); it sizes the neighbour-search grids only, never a result.  A cloud
    with fewer than ``ransac_n`` points is returned as it is (the engine's floor-skip rule), and a band of fewer than
    ``ransac_n`` points has no plane (nothing is removed from it).  Returns a list of ``PointCloud``."""
    from .pipeline import FramePipeline, PipelineConfig
    if nb_neighbors < 1 or not std_ratio > 0:
        raise _cabi.KinectPyB200Error(_cabi.KP_E_ARG, "nb_neighbors < 1 or std_ratio <= 0")
    pcds = list(pcds)
    if not pcds:
        return []
    cap = max(max(len(p) for p in pcds), 1)
    cfg = PipelineConfig(input_mode=_cabi.INPUT_CLOUDS, cloud_voxel=0, n_sensors=1, pixels=cap, scale=1.0, voxel_size=float(spacing),
                         sor_k=0, do_floor=True, floor_band=float(band), ransac_thr=float(distance_threshold),
                         ransac_n=int(ransac_n), ransac_iters=int(num_iterations), floor_sor_k=int(nb_neighbors),
                         floor_sor_ratio=float(std_ratio), do_icp=False, n_streams=int(n_streams),
                         seed=int(geometry._SEED[0] if seed is None else seed) & 0xFFFFFFFFFFFFFFFF)
    pipe = FramePipeline(cfg)
    try:
        outs = pipe.run_clouds(pcds, want_points=True, out_stride=cap)
    finally:
        pipe.close()
    return [PointCloud(o.points) for o in outs]


def main(pattern='E:/Extracted_data/*/*/*/master_1/filtered_and_registered_pointclouds/*.pcd'):
    for i, fp in enumerate(glob.glob(pattern)):
        if i % 100 == 0:
            print(i)
        filtered = remove_floor(read_point_cloud(fp))
        dst = fp.replace('filtered_and_registered_pointclouds', 'floor_filter_and_registered_pointclouds')
        os.makedirs(os.path.dirname(dst), exist_ok=True)   # the reference mkdirs the file path itself (SURVEY.md App. B)
        write_point_cloud(dst, filtered)


if __name__ == '__main__':
    main()
