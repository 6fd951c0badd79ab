#!/usr/bin/env python
"""Generate tests/golden/reference_compositions.npz and reference_registrations.npz by RUNNING THE REFERENCE'S OWN
WRAPPERS (a checkout of tiborcamargo/KinectPy, read-only).

Open3D is absent here, so the reference's wrapper code is executed, unmodified, against an ``open3d`` stand-in
whose geometry routines are the CPU oracle's (oracle/kp_oracle.c).  What this pins is everything the WRAPPERS
decide -- which routine is called on which cloud, in which order, with which arguments and defaults, what is
copied and what is returned:

* ``preprocessing.filtering.filter_outliers``                         (preprocessing/filtering.py:12-25)
* ``preprocessing.registration.execute_point_to_plane_registration`` (preprocessing/registration.py:65-86, through
  ``prepare_dataset`` / ``preprocess_point_cloud`` :7-29 -- note the double source/target swap)
* the floor-removal body of ``floor_removal.py`` (:63-73), exec'd verbatim from the file's own source lines
* the fusion body of ``DataProcessor``'s frame loop (preprocessing/data.py:41-61), exec'd verbatim likewise
* ``utils.processing.statistical_outlier_removal``                    (utils/processing.py:302-310)
* ``preprocessing.registration.execute_global_registration``         (preprocessing/registration.py:32-62)
* ``preprocessing.registration.execute_colored_ICP_registration``    (preprocessing/registration.py:89-114)

tests/test_golden.py then checks that the oracle's array-level compositions (``oracle.filter_outliers``,
``oracle.remove_floor``, and the registration composition the frame pipeline uses) reproduce these outputs;
the GPU tests compare the kernels with those compositions.

Run:  python tests/golden/make_composition_golden.py <KinectPy checkout>     (the .npz files are committed)
"""
import contextlib
import copy
import io
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "reference_compositions.npz")
OUT_REG = os.path.join(HERE, "reference_registrations.npz")      # glob_* / col_*: kept apart so each file stays under 1 MB
sys.path.insert(0, ROOT)

CALLS = []          # (routine, arguments) in the order the reference's wrappers made them


def oracle_backed_namespace():
    """(PointCloud, registration namespace, geometry namespace): the slice of Open3D the wrappers touch, computed by the oracle."""
    from oracle import oracle as orc

    class PointCloud:
        def __init__(self, points=None):
            self.points = np.zeros((0, 3)) if points is None else np.asarray(points, dtype=np.float64)
            self.colors = np.zeros((0, 3))
            self.normals = np.zeros((0, 3))

        def has_normals(self):
            return len(self.normals) == len(self.points) and len(self.points) > 0

        def voxel_down_sample(self, voxel_size):
            CALLS.append(("voxel_down_sample", float(voxel_size), len(self.points)))
            has_c = len(self.colors) == len(self.points) and len(self.points) > 0
            v = orc.voxel_downsample(self.points, float(voxel_size), colors=self.colors if has_c else None)
            out = PointCloud(v["points"])
            if has_c:
                out.colors = v["colors"].astype(np.float64)
            return out

        def remove_statistical_outlier(self, nb_neighbors, std_ratio):
            CALLS.append(("remove_statistical_outlier", int(nb_neighbors), float(std_ratio), len(self.points)))
            keep, _, _ = orc.sor(self.points, int(nb_neighbors), float(std_ratio))
            idx = np.flatnonzero(keep)
            return self.select_by_index(idx), idx.tolist()

        def estimate_normals(self, search_param):
            CALLS.append(("estimate_normals", float(search_param.radius), int(search_param.max_nn), len(self.points)))
            self.normals = orc.estimate_normals(self.points, float(search_param.radius), int(search_param.max_nn)).astype(np.float64)

        def segment_plane(self, distance_threshold, ransac_n, num_iterations):
            CALLS.append(("segment_plane", float(distance_threshold), int(ransac_n), int(num_iterations), len(self.points)))
            plane, mask, _, _ = orc.ransac_plane(self.points, float(distance_threshold), int(ransac_n), int(num_iterations),
                                                 seed=1234)
            return plane, np.flatnonzero(mask).tolist()

        def select_by_index(self, indices, invert=False):
            idx = np.asarray(indices, dtype=np.int64).reshape(-1)
            mask = np.zeros(len(self.points), dtype=bool)
            mask[idx] = True
            if invert:
                mask = ~mask
            out = PointCloud(np.asarray(self.points)[mask])
            if self.has_normals():
                out.normals = np.asarray(self.normals)[mask]
            return out

        def transform(self, T):
            CALLS.append(("transform", np.asarray(T, np.float64).round(12).tolist(), len(self.points)))
            self.points = orc.transform(self.points, T).astype(np.float64)
            return self

        def __add__(self, other):
            return PointCloud(np.concatenate([np.asarray(self.points), np.asarray(other.points)], axis=0))

    class Hybrid:
        def __init__(self, radius, max_nn):
            self.radius, self.max_nn = radius, max_nn

    class PointToPlane:
        pass

    class Result:
        pass

    def registration_icp(source, target, threshold, init, estimation, *rest):
        assert isinstance(estimation, PointToPlane) and target.has_normals()
        CALLS.append(("registration_icp", float(threshold), len(source.points), len(target.points)))
        r = orc.icp_point_to_plane(source.points, target.points, target.normals, float(threshold), init=init, max_iter=30)
        out = Result()
        out.transformation, out.fitness, out.inlier_rmse = r["T"], r["fitness"], r["rmse"]
        return out

    class Feature:
        def __init__(self, rows):
            self.rows = rows                    # [n, 33]
            self.data = rows.T                  # Open3D's layout

    def compute_fpfh_feature(pcd, search_param):
        CALLS.append(("compute_fpfh_feature", float(search_param.radius), int(search_param.max_nn), len(pcd.points)))
        return Feature(orc.fpfh(pcd.points, pcd.normals, float(search_param.radius), int(search_param.max_nn)))

    class PointToPoint:
        def __init__(self, with_scaling=False):
            self.with_scaling = with_scaling

    class EdgeLength:
        def __init__(self, similarity_threshold=0.9):
            self.similarity_threshold = similarity_threshold

    class Distance:
        def __init__(self, distance_threshold):
            self.distance_threshold = distance_threshold

    class RansacCriteria:
        def __init__(self, max_iteration=100000, confidence=0.999):
            self.max_iteration, self.confidence = max_iteration, confidence

    class IcpCriteria:
        def __init__(self, relative_fitness=1e-6, relative_rmse=1e-6, max_iteration=30):
            self.relative_fitness, self.relative_rmse, self.max_iteration = relative_fitness, relative_rmse, max_iteration

    class ColoredIcp:
        pass

    ransac_calls = [0]

    def registration_ransac_based_on_feature_matching(source, target, sf, tf, mutual_filter, max_corr, estimation, ransac_n,
                                                      checkers, criteria):
        assert isinstance(estimation, PointToPoint) and estimation.with_scaling is False
        assert isinstance(checkers[0], EdgeLength) and isinstance(checkers[1], Distance)
        CALLS.append(("registration_ransac_based_on_feature_matching", bool(mutual_filter), float(max_corr), int(ransac_n),
                      float(checkers[0].similarity_threshold), float(checkers[1].distance_threshold),
                      int(criteria.max_iteration), float(criteria.confidence), len(source.points), len(target.points)))
        nn_st, _ = orc.feature_match(sf.rows, tf.rows)
        nn_ts, _ = orc.feature_match(tf.rows, sf.rows)
        cor = orc.mutual_correspondences(nn_st, nn_ts, bool(mutual_filter), int(ransac_n))
        # successive calls draw from successive streams, as successive upstream calls advance the global generator
        seed = (1234 + 0x9E3779B97F4A7C15 * ransac_calls[0]) & 0xFFFFFFFFFFFFFFFF
        ransac_calls[0] += 1
        r = orc.ransac_correspondence(source.points, target.points, cor, float(max_corr), int(ransac_n),
                                      float(checkers[0].similarity_threshold), float(checkers[1].distance_threshold),
                                      int(criteria.max_iteration), float(criteria.confidence), seed=seed)
        out = Result()
        out.transformation, out.fitness, out.inlier_rmse = r["T"], r["fitness"], r["rmse"]
        return out

    def registration_colored_icp(source, target, max_corr, init, estimation, criteria):
        assert isinstance(estimation, ColoredIcp) and target.has_normals()
        CALLS.append(("registration_colored_icp", float(max_corr), int(criteria.max_iteration), float(criteria.relative_fitness),
                      float(criteria.relative_rmse), len(source.points), len(target.points)))
        r = orc.icp_colored(source.points, source.colors, target.points, target.colors, target.normals, float(max_corr),
                            init=init, max_iter=int(criteria.max_iteration), rel_fit=float(criteria.relative_fitness),
                            rel_rmse=float(criteria.relative_rmse))
        out = Result()
        out.transformation, out.fitness, out.inlier_rmse = r["T"], r["fitness"], r["rmse"]
        return out

    registration = types.SimpleNamespace(
        registration_icp=registration_icp, TransformationEstimationPointToPlane=PointToPlane,
        compute_fpfh_feature=compute_fpfh_feature, TransformationEstimationPointToPoint=PointToPoint,
        CorrespondenceCheckerBasedOnEdgeLength=EdgeLength, CorrespondenceCheckerBasedOnDistance=Distance,
        RANSACConvergenceCriteria=RansacCriteria, ICPConvergenceCriteria=IcpCriteria,
        TransformationEstimationForColoredICP=ColoredIcp,
        registration_ransac_based_on_feature_matching=registration_ransac_based_on_feature_matching,
        registration_colored_icp=registration_colored_icp, _ransac_calls=ransac_calls)
    geometry = types.SimpleNamespace(PointCloud=PointCloud, KDTreeSearchParamHybrid=Hybrid)
    return PointCloud, registration, geometry


def install_oracle_backed_open3d():
    PointCloud, registration, geometry = oracle_backed_namespace()
    o3d = types.ModuleType("open3d")
    o3d.geometry = geometry
    o3d.utility = types.SimpleNamespace(Vector3dVector=lambda a: np.asarray(a, dtype=np.float64))
    o3d.pipelines = types.SimpleNamespace(registration=registration)
    o3d.visualization = types.SimpleNamespace()
    o3d.io = types.SimpleNamespace()
    sys.modules["open3d"] = o3d
    for name in ("tensorflow", "imghdr", "PIL", "PIL.Image", "cv2"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["PIL"].Image = sys.modules["PIL.Image"]
    return PointCloud


def scene(n, seed, mm=False):
    """A floor (y = max), a wall and a blob standing on the floor, plus a few stray points; metres or millimetres."""
    r = np.random.default_rng(seed)
    floor = np.stack([r.uniform(-1, 1, n // 2), 1.2 + r.normal(0, 0.002, n // 2), r.uniform(1, 3, n // 2)], 1)
    wall = np.stack([r.uniform(-1, 1, n // 4), r.uniform(-0.8, 1.2, n // 4), 3.0 + r.normal(0, 0.002, n // 4)], 1)
    blob = r.normal(0, 0.12, (n // 4, 3)) * [1, 3, 1] + [0, 0.7, 2.0]
    blob[:, 1] = np.minimum(blob[:, 1], 1.19)          # it stands on the floor, nothing lies below it
    stray = r.uniform(-1, 1, (n // 100, 3)) + [0, 0, 2]
    pts = np.concatenate([floor, wall, blob, stray], 0)
    return (pts * (1000.0 if mm else 1.0)).astype(np.float32)


def main():
    ref = sys.argv[1]          # a checkout of tiborcamargo/KinectPy
    PointCloud = install_oracle_backed_open3d()
    sys.path.insert(0, ref)
    from preprocessing import filtering as ref_filtering
    from preprocessing import registration as ref_registration
    out = {}

    # ---- filter_outliers: explicit arguments (BASELINE config 1) and the reference's defaults (units: metres / mm)
    pts = scene(6000, 1)
    del CALLS[:]
    got = ref_filtering.filter_outliers(PointCloud(pts), nb_neighbors=20, std_ratio=2.0, voxel_size=0.02)
    out["fo_in"], out["fo_out"] = pts, np.asarray(got.points, np.float32)
    out["fo_calls"] = np.array(repr(CALLS))
    pts_mm = scene(6000, 2, mm=True)
    del CALLS[:]
    src = PointCloud(pts_mm)
    got = ref_filtering.filter_outliers(src)          # defaults 200 / 3.0 / 0.02: on mm data every point is its own voxel
    out["fo_default_in"], out["fo_default_out"] = pts_mm, np.asarray(got.points, np.float32)
    out["fo_default_calls"] = np.array(repr(CALLS))
    assert np.array_equal(np.asarray(src.points, np.float32), pts_mm)       # the input cloud is not modified

    # ---- execute_point_to_plane_registration (mm units, the reference's voxel 35 / threshold 100)
    from kinectpy_b200 import synth
    master = scene(8000, 3, mm=True)
    D = synth.perturbed_extrinsic(np.eye(4), angle_deg=1.0, shift_mm=(12, -8, 10), unit_scale=1.0)
    from oracle import oracle as orc
    sub = orc.transform(scene(8000, 4, mm=True), np.linalg.inv(D))
    init = np.eye(4)
    del CALLS[:]
    with contextlib.redirect_stdout(io.StringIO()):
        T = ref_registration.execute_point_to_plane_registration(PointCloud(master), PointCloud(sub), init, voxel_size=35)
    out["reg_master"], out["reg_sub"], out["reg_init"], out["reg_T"] = master, sub, init, np.asarray(T, np.float64)
    out["reg_calls"] = np.array(repr(CALLS))
    # the wrappers' own source text (fixture data, like floor_source / fuse_source below): tests/test_gpu_dropin.py executes
    # it, unmodified, over kinectpy_b200.o3d without a KinectPy checkout
    import inspect
    out["fo_source"] = np.array(inspect.getsource(ref_filtering.filter_outliers))
    out["reg_source"] = np.array("\n".join(inspect.getsource(f) for f in (ref_registration.preprocess_point_cloud, ref_registration.prepare_dataset,
                                                                          ref_registration.execute_point_to_plane_registration)))

    # ---- floor removal: the body of the script's loop, exec'd verbatim from the reference's file
    src_lines = open(os.path.join(ref, "floor_removal.py")).read().splitlines()
    main_at = next(i for i, ln in enumerate(src_lines) if ln.startswith("if __name__"))
    first = next(i for i, ln in enumerate(src_lines) if i > main_at and "pcd_points = np.asarray(pcd.points)" in ln)
    last = next(i for i, ln in enumerate(src_lines) if i > main_at and "remove_statistical_outlier(" in ln)
    body = "\n".join(ln[8:] if ln.startswith(" " * 8) else ln.strip() for ln in src_lines[first:last + 1])
    floor_in = scene(9000, 5, mm=True)
    ns = {"np": np, "pcd": PointCloud(floor_in)}
    del CALLS[:]
    exec(body, ns)
    out["floor_in"] = floor_in
    out["floor_out"] = np.asarray(ns["filtered_pcd"].points, np.float32)
    out["floor_plane"] = np.asarray(ns["plane_model"], np.float64)
    out["floor_inliers"] = np.asarray(ns["inliers"], np.int64)
    out["floor_calls"] = np.array(repr(CALLS))
    out["floor_source"] = np.array(body)

    # ---- fusion: the body of DataProcessor's frame loop (preprocessing/data.py:41-61), exec'd verbatim
    from preprocessing import data as ref_data        # (only for its module-level imports to resolve as in the reference)
    del ref_data
    src_lines = open(os.path.join(ref, "preprocessing", "data.py")).read().splitlines()
    first = next(i for i, ln in enumerate(src_lines) if "registered_pcd_points, registered_pcd_colors = [], []" in ln)
    last = next(i for i, ln in enumerate(src_lines) if "registered_pcd = filter_outliers(registered_pcd)" in ln)
    body = "\n".join(ln[12:] if ln.startswith(" " * 12) else ln.strip() for ln in src_lines[first:last + 1])
    clouds = [scene(3000, 10 + s) for s in range(3)]
    Ts = [synth.perturbed_extrinsic(np.eye(4), angle_deg=20.0 * (s + 1), shift_mm=(300, -100, 200), unit_scale=1e-3) for s in range(2)]
    pcs = [PointCloud(c) for c in clouds]
    for pc in pcs:
        pc.colors = np.full((len(pc.points), 3), 0.5)
    ns = {"np": np, "o3d": sys.modules["open3d"], "filter_outliers": ref_filtering.filter_outliers, "filtered_pcds": pcs,
          "self": types.SimpleNamespace(registration_transformations=Ts)}
    del CALLS[:]
    exec(body, ns)
    out["fuse_in"] = np.stack(clouds)
    out["fuse_T"] = np.stack(Ts)
    out["fuse_out"] = np.asarray(ns["registered_pcd"].points, np.float32)
    out["fuse_calls"] = np.array(repr(CALLS))
    out["fuse_source"] = np.array(body)

    # ---- utils.processing.statistical_outlier_removal (utils/processing.py:302-310): hard-coded 0.02 voxel
    from utils import processing as ref_processing
    so_in = scene(5000, 20)
    del CALLS[:]
    got = ref_processing.statistical_outlier_removal(PointCloud(so_in))
    out["so_in"], out["so_out"] = so_in, np.asarray(got.points, np.float32)
    out["so_calls"] = np.array(repr(CALLS))

    # ---- execute_global_registration (registration.py:32-62): 15 trials, each re-running prepare_dataset
    reg_ns = sys.modules["open3d"].pipelines.registration
    gm = scene(3000, 30, mm=True)
    Dg = synth.perturbed_extrinsic(np.eye(4), angle_deg=25.0, shift_mm=(300, -150, 200), unit_scale=1.0)
    gs = orc.transform(gm, np.linalg.inv(Dg))
    del CALLS[:]
    reg_ns._ransac_calls[0] = 0
    Tg = ref_registration.execute_global_registration(PointCloud(gm), PointCloud(gs), voxel_size=60, ransac_n_trials=3)
    out["glob_master"], out["glob_sub"], out["glob_T"] = gm, gs, np.asarray(Tg, np.float64)
    out["glob_calls"] = np.array(repr(CALLS))
    assert np.abs(out["glob_T"] - Dg)[:3, :3].max() < 0.05, "the planted transform is recovered"

    # ---- execute_colored_ICP_registration (registration.py:89-114): three scales, each from the initial transform
    cm = scene(6000, 31, mm=True)
    ccol = (0.5 + 0.5 * np.sin(cm / 90.0)).astype(np.float32)          # a smooth texture
    Dc = synth.perturbed_extrinsic(np.eye(4), angle_deg=0.8, shift_mm=(10, -6, 8), unit_scale=1.0)
    cs = orc.transform(cm, np.linalg.inv(Dc))
    pm, ps = PointCloud(cm), PointCloud(cs)
    pm.colors, ps.colors = ccol.astype(np.float64), ccol.astype(np.float64)
    del CALLS[:]
    Tc = ref_registration.execute_colored_ICP_registration(pm, ps, np.eye(4))
    out["col_master"], out["col_sub"], out["col_colors"], out["col_T"] = cm, cs, ccol, np.asarray(Tc, np.float64)
    out["col_calls"] = np.array(repr(CALLS))

    reg = {k: out[k] for k in out if k.startswith(("glob_", "col_"))}
    np.savez_compressed(OUT, **{k: v for k, v in out.items() if k not in reg})
    np.savez_compressed(OUT_REG, **reg)
    for k in ("fo_calls", "fo_default_calls", "reg_calls", "floor_calls", "fuse_calls", "so_calls", "glob_calls", "col_calls"):
        print(k, out[k])
    print("wrote", OUT, {k: getattr(v, "shape", None) for k, v in out.items()})


if __name__ == "__main__":
    main()
