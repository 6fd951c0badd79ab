"""numpy front-end of the CPU oracle (``oracle/kp_oracle.c``).

TEST INFRASTRUCTURE ONLY -- imported by ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py``; never by ``kinectpy_b200``.
PARITY UNPINNED against Open3D (absent from this image, no golden vectors in the reference): see
the header of ``kp_oracle.c``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libkp_oracle.so")
_lib = None

F_INT16 = 1
F_DROP_ANY_ZERO = 2


def build(force: bool = False) -> str:
    """Compile the C restatement with gcc (no FMA contraction, OpenMP if available).  In a tree that cannot be
    written (a read-only checkout) the library goes to a temporary directory instead."""
    global _SO
    src = os.path.join(_HERE, "kp_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        try:
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            writable = os.access(os.path.dirname(_SO), os.W_OK)
        except OSError:
            writable = False
        if not writable:
            _SO = os.path.join(tempfile.mkdtemp(prefix="kp_oracle_"), "libkp_oracle.so")
        base = ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-fvisibility=hidden", "-o", _SO, src, "-lm"]
        for cc in ("/usr/bin/gcc", "gcc", "cc"):
            for omp in (["-fopenmp"], []):
                try:
                    subprocess.run([cc] + omp + base, check=True, capture_output=True)
                    return _SO
                except (subprocess.CalledProcessError, FileNotFoundError):
                    continue
        raise RuntimeError("could not compile oracle/kp_oracle.c")
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.kpo_rng.restype = C.c_uint64
        _lib.kpo_rng.argtypes = [C.c_uint64] * 3
        _lib.kpo_csum.restype = C.c_double
        _lib.kpo_csum.argtypes = [C.c_void_p, C.c_long]
        _lib.kpo_voxel_downsample.restype = C.c_long
        _lib.kpo_sor.restype = C.c_long
        _lib.kpo_radius_outlier.restype = C.c_long
        _lib.kpo_ransac_plane.restype = C.c_long
        _lib.kpo_plane_side.restype = C.c_long
        _lib.kpo_num_threads.restype = C.c_int
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def num_threads() -> int:
    return int(lib().kpo_num_threads())


def set_num_threads(n: int) -> None:
    """OpenMP threads of the oracle's loops (torchrun exports OMP_NUM_THREADS=1 to its workers)."""
    lib().kpo_set_num_threads(C.c_int(int(n)))


def rng(seed, a, b) -> int:
    return int(lib().kpo_rng(C.c_uint64(seed), C.c_uint64(a), C.c_uint64(b)))


def _mix64_np(z):
    z = (z + np.uint64(0x9E3779B97F4A7C15))
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def rng_array(seed, a, b):
    """kp_rng(seed, a, b[i]) for an index array b (vectorised restatement of kpo_rng)."""
    with np.errstate(over="ignore"):
        s = _mix64_np(np.uint64(seed & 0xFFFFFFFFFFFFFFFF))
        s = _mix64_np(s + np.uint64(a & 0xFFFFFFFFFFFFFFFF))
        return _mix64_np(s + np.asarray(b, dtype=np.uint64))


def resample_fixed_n(pts, N, mode="random", seed=1234, stream=0):
    """Fixed-N resampling (select_points_randomly, utils/processing.py:259-275; points[:N],
    datasets/kinect_dataset_npz.py:97).  Random mode: the N valid points with the smallest
    (key, index), key = min(rng(seed, stream, i) >> 32, 2^32 - 2), NaN rows excluded; ValueError when
    fewer than N valid points exist (np.random.choice(replace=False) raises it).  Returns (points, indices)."""
    pts = _f32(pts).reshape(-1, 3)
    n = pts.shape[0]
    if mode == "prefix":
        m = min(n, int(N))
        return pts[:m].copy(), np.arange(m, dtype=np.int32)
    key = (rng_array(seed, stream, np.arange(n, dtype=np.uint64)) >> np.uint64(32)).astype(np.uint64)
    key = np.minimum(key, np.uint64(0xFFFFFFFE))
    valid = ~np.isnan(pts[:, 0])
    key[~valid] = np.uint64(0xFFFFFFFF)
    if int(N) > int(valid.sum()):
        raise ValueError("Cannot take a larger sample than population when 'replace=False'")
    order = np.argsort(key, kind="stable")[:int(N)].astype(np.int32)
    return pts[order].copy(), order


def csum(x) -> float:
    x = np.ascontiguousarray(x, dtype=np.float64)
    return float(lib().kpo_csum(_p(x), C.c_long(x.size)))


def unproject(depth, xytab, T=None, flags=0, scale=1e-3, want_xyz16=False):
    """depth uint16[B,S,P], xytab float32[S,P,2], T float64[S,4,4] -> xyz float32[B,S*P,3], valid, xyz16."""
    depth = np.ascontiguousarray(depth, dtype=np.uint16)
    B, S, P = depth.shape
    xytab = _f32(xytab).reshape(S, P, 2)
    Tc = None if T is None else np.ascontiguousarray(T, dtype=np.float64).reshape(S, 16)
    xyz = np.empty((B, S * P, 3), dtype=np.float32)
    valid = np.empty((B, S * P), dtype=np.uint8)
    xyz16 = np.zeros((B, S * P, 3), dtype=np.int16) if want_xyz16 else None
    lib().kpo_unproject(_p(depth), _p(xytab), _p(Tc), C.c_int(B), C.c_int(S), C.c_long(P), C.c_int(flags),
                        C.c_double(scale), _p(xyz), _p(valid), _p(xyz16))
    return xyz, valid, xyz16


def points_from_xyz16(xyz16, T=None, flags=F_DROP_ANY_ZERO, scale=1.0, keep=None):
    """utils/io.py:29-41 restated: int16 [n,3] -> float32 points (NaN where invalid) and validity."""
    a = np.asarray(xyz16, dtype=np.int16).reshape(-1, 3)
    X = a.astype(np.float64) * scale
    ok = np.ones(a.shape[0], dtype=bool)
    if flags & F_DROP_ANY_ZERO:
        ok &= (X[:, 0] != 0) & (X[:, 1] != 0) & (X[:, 2] != 0)
    if keep is not None:
        ok &= np.asarray(keep).reshape(-1) != 0
    if T is not None:
        M = np.asarray(T, dtype=np.float64).reshape(4, 4)
        x, y, z = X[:, 0], X[:, 1], X[:, 2]
        X = np.stack([((M[r, 0] * x + M[r, 1] * y) + M[r, 2] * z) + M[r, 3] for r in range(3)], axis=1)
    out = X.astype(np.float32)
    out[~ok] = np.nan
    return out, ok.astype(np.uint8)


def crop_mask(rgb, xyz16, gate=750.0):
    """preprocessing/data.py:165-178 restated (numpy is what the reference itself uses here)."""
    rgb = np.asarray(rgb).reshape(-1, 3)
    z = np.asarray(xyz16).reshape(-1, 3)[:, 2]
    med = np.median(z)
    valid_pixels = (rgb[:, 0] != 0) & (rgb[:, 1] != 0) & (rgb[:, 2] != 0)
    valid_depths = (z <= med + gate) | (z <= med - gate)
    return (valid_pixels & valid_depths).astype(np.uint8), float(med)


def transform(xyz, T, rotate_only=False):
    out = _f32(xyz).copy()
    M = np.ascontiguousarray(T, dtype=np.float64).reshape(16)
    lib().kpo_transform(_p(out), C.c_long(out.shape[0]), _p(M), C.c_int(1 if rotate_only else 0))
    return out


def voxel_downsample(xyz, voxel, colors=None, normals=None):
    xyz = _f32(xyz)
    n = xyz.shape[0]
    colors = None if colors is None else _f32(colors)
    normals = None if normals is None else _f32(normals)
    o_p = np.empty((max(n, 1), 3), np.float32)
    o_c = np.empty((max(n, 1), 3), np.float32) if colors is not None else None
    o_n = np.empty((max(n, 1), 3), np.float32) if normals is not None else None
    ijk = np.empty((max(n, 1), 3), np.int32)
    pv = np.empty((max(n, 1),), np.int32)
    minb = np.zeros(3, np.float64)
    m = lib().kpo_voxel_downsample(_p(xyz), _p(colors), _p(normals), C.c_long(n), C.c_double(voxel), _p(o_p), _p(o_c),
                                   _p(o_n), _p(ijk), _p(pv), _p(minb))
    if m < 0:
        raise ValueError(f"oracle voxel_downsample failed ({m})")
    return {"points": o_p[:m], "colors": None if o_c is None else o_c[:m], "normals": None if o_n is None else o_n[:m],
            "ijk": ijk[:m], "point_voxel": pv[:n], "min_bound": minb, "m": int(m)}


def knn(pts, k, queries=None, radius=0.0):
    pts = _f32(pts)
    q = None if queries is None else _f32(queries)
    nq = pts.shape[0] if q is None else q.shape[0]
    idx = np.empty((nq, k), np.int32)
    d2 = np.empty((nq, k), np.float64)
    cnt = np.empty((nq,), np.int32)
    lib().kpo_knn(_p(pts), C.c_long(pts.shape[0]), _p(q), C.c_long(nq), C.c_int(k), C.c_double(radius), _p(idx), _p(d2),
                  _p(cnt))
    return idx, d2, cnt


def sor(pts, k, std_ratio, cell_hint=0.0):
    pts = _f32(pts)
    n = pts.shape[0]
    keep = np.zeros((n,), np.uint8)
    mean = np.zeros((n,), np.float64)
    stats = np.zeros(3, np.float64)
    kept = lib().kpo_sor(_p(pts), C.c_long(n), C.c_int(k), C.c_double(std_ratio), C.c_double(cell_hint), _p(keep),
                         _p(mean), _p(stats))
    if kept < 0:
        raise ValueError("oracle sor: bad arguments")
    return keep, mean, stats


def radius_outlier(pts, nb_points, radius):
    pts = _f32(pts)
    n = pts.shape[0]
    keep = np.zeros((n,), np.uint8)
    counts = np.zeros((n,), np.int32)
    kept = lib().kpo_radius_outlier(_p(pts), C.c_long(n), C.c_int(nb_points), C.c_double(radius), _p(keep), _p(counts))
    if kept < 0:
        raise ValueError("oracle radius_outlier: bad arguments")
    return keep, counts


def estimate_normals(pts, radius, max_nn):
    pts = _f32(pts)
    out = np.zeros_like(pts)
    lib().kpo_estimate_normals(_p(pts), C.c_long(pts.shape[0]), C.c_double(radius), C.c_int(max_nn), _p(out))
    return out


def smallest_eigvec(cov6):
    c = np.ascontiguousarray(cov6, dtype=np.float64)
    out = np.zeros(3)
    lib().kpo_smallest_eigvec(_p(c), _p(out))
    return out


def ransac_sample(seed, h, n, ransac_n):
    ids = np.zeros(ransac_n, np.int64)
    lib().kpo_ransac_sample(C.c_uint64(seed), C.c_long(h), C.c_long(n), C.c_int(ransac_n), _p(ids))
    return ids


def ransac_plane(pts, thr, ransac_n, iters, probability=0.99999999, seed=1234):
    pts = _f32(pts)
    n = pts.shape[0]
    plane = np.zeros(4, np.float64)
    mask = np.zeros((n,), np.uint8)
    best = C.c_int32(-1)
    counts = np.zeros((iters,), np.int64)
    ninl = lib().kpo_ransac_plane(_p(pts), C.c_long(n), C.c_double(thr), C.c_int(ransac_n), C.c_int(iters),
                                  C.c_double(probability), C.c_uint64(seed), _p(plane), _p(mask), C.byref(best),
                                  _p(counts))
    if ninl < 0:
        raise ValueError("oracle ransac_plane: bad arguments")
    return plane, mask, int(best.value), counts


def plane_side(pts, a, b, c, d):
    pts = _f32(pts)
    keep = np.zeros((pts.shape[0],), np.uint8)
    lib().kpo_plane_side(_p(pts), C.c_long(pts.shape[0]), C.c_double(a), C.c_double(b), C.c_double(c), C.c_double(d),
                         _p(keep))
    return keep


def band_mask(pts, band, axis=1):
    """floor_removal.py:64-66 restated: lower = coord >= max(coord) - band (float64 compare)."""
    v = np.asarray(pts, dtype=np.float32)[:, axis].astype(np.float64)
    return (v >= v.max() - band).astype(np.uint8)


def icp_point_to_plane(src, tgt, tgt_normals, max_corr, init=None, max_iter=30, rel_fit=1e-6, rel_rmse=1e-6):
    src, tgt, tn = _f32(src), _f32(tgt), _f32(tgt_normals)
    T0 = np.ascontiguousarray(np.eye(4) if init is None else init, dtype=np.float64).reshape(16)
    T = np.zeros(16, np.float64)
    fit, rmse, iters, nc = C.c_double(), C.c_double(), C.c_int(), C.c_int64()
    rc = lib().kpo_icp_point_to_plane(_p(src), C.c_long(src.shape[0]), _p(tgt), _p(tn), C.c_long(tgt.shape[0]),
                                      C.c_double(max_corr), _p(T0), C.c_int(max_iter), C.c_double(rel_fit),
                                      C.c_double(rel_rmse), _p(T), C.byref(fit), C.byref(rmse), C.byref(iters), C.byref(nc))
    if rc != 0:
        raise ValueError("oracle icp: bad arguments")
    return {"T": T.reshape(4, 4), "fitness": fit.value, "rmse": rmse.value, "iters": iters.value, "ncorr": nc.value}


def umeyama(src, tgt):
    """TransformationEstimationPointToPoint.compute_transformation on matched rows (manual_pointcloud_registration.py:90-92)."""
    a = np.ascontiguousarray(src, dtype=np.float64).reshape(-1, 3)
    b = np.ascontiguousarray(tgt, dtype=np.float64).reshape(-1, 3)
    T = np.zeros(16, np.float64)
    lib().kpo_umeyama(_p(a), _p(b), C.c_long(a.shape[0]), _p(T))
    return T.reshape(4, 4)


def color_gradient(pts, colors, normals, radius, max_nn=30):
    """(intensity, gradient) of InitializePointCloudForColoredICP (under registration_colored_icp, registration.py:108)."""
    pts, col, nrm = _f32(pts), _f32(colors), _f32(normals)
    n = pts.shape[0]
    inten = np.zeros((n,), np.float32)
    grad = np.zeros((n, 3), np.float32)
    if lib().kpo_color_gradient(_p(pts), _p(col), _p(nrm), C.c_long(n), C.c_double(radius), C.c_int(max_nn), _p(inten), _p(grad)) != 0:
        raise ValueError("oracle color_gradient: bad arguments")
    return inten, grad


def _icp(mode, src, tgt, tgt_normals, src_int, tgt_int, tgt_grad, lam, max_corr, init, max_iter, rel_fit, rel_rmse):
    src, tgt = _f32(src), _f32(tgt)
    tn = None if tgt_normals is None else _f32(tgt_normals)
    T0 = np.ascontiguousarray(np.eye(4) if init is None else init, dtype=np.float64).reshape(16)
    T = np.zeros(16, np.float64)
    fit, rmse, iters, nc = C.c_double(), C.c_double(), C.c_int(), C.c_int64()
    rc = lib().kpo_icp(C.c_int(mode), _p(src), C.c_long(src.shape[0]), _p(tgt), _p(tn), C.c_long(tgt.shape[0]),
                       _p(src_int), _p(tgt_int), _p(tgt_grad), C.c_double(lam), C.c_double(max_corr), _p(T0), C.c_int(max_iter),
                       C.c_double(rel_fit), C.c_double(rel_rmse), _p(T), C.byref(fit), C.byref(rmse), C.byref(iters), C.byref(nc))
    if rc != 0:
        raise ValueError("oracle icp: bad arguments")
    return {"T": T.reshape(4, 4), "fitness": fit.value, "rmse": rmse.value, "iters": iters.value, "ncorr": nc.value}


def icp_point_to_point(src, tgt, max_corr, init=None, max_iter=30, rel_fit=1e-6, rel_rmse=1e-6):
    """registration_icp(..., TransformationEstimationPointToPoint()) (manual_pointcloud_registration.py:94-98)."""
    return _icp(1, src, tgt, None, None, None, None, 1.0, max_corr, init, max_iter, rel_fit, rel_rmse)


def icp_colored(src, src_colors, tgt, tgt_colors, tgt_normals, max_corr, init=None, max_iter=30, rel_fit=1e-6,
                rel_rmse=1e-6, lambda_geometric=0.968):
    """registration_colored_icp (preprocessing/registration.py:108-113)."""
    sc = _f32(src_colors)
    s_int = ((sc[:, 0].astype(np.float64) + sc[:, 1].astype(np.float64)) + sc[:, 2].astype(np.float64)) / 3.0
    s_int = s_int.astype(np.float32)
    t_int, t_grad = color_gradient(tgt, tgt_colors, tgt_normals, 2.0 * max_corr, 30)
    return _icp(2, src, tgt, tgt_normals, s_int, t_int, t_grad, lambda_geometric, max_corr, init, max_iter, rel_fit, rel_rmse)


def fpfh(pts, normals, radius, max_nn):
    """compute_fpfh_feature (preprocessing/registration.py:17-20): float64 [n, 33]."""
    pts, nrm = _f32(pts), _f32(normals)
    feat = np.zeros((pts.shape[0], 33), np.float64)
    if lib().kpo_fpfh(_p(pts), _p(nrm), C.c_long(pts.shape[0]), C.c_double(radius), C.c_int(max_nn), _p(feat)) != 0:
        raise ValueError("oracle fpfh: bad arguments")
    return feat


def feature_match(fa, fb):
    fa = np.ascontiguousarray(fa, dtype=np.float64)
    fb = np.ascontiguousarray(fb, dtype=np.float64)
    nn = np.zeros((fa.shape[0],), np.int32)
    d2 = np.zeros((fa.shape[0],), np.float64)
    lib().kpo_feature_match(_p(fa), C.c_long(fa.shape[0]), _p(fb), C.c_long(fb.shape[0]), C.c_int(fa.shape[1]), _p(nn), _p(d2))
    return nn, d2


def mutual_correspondences(nn_st, nn_ts, mutual_filter=True, ransac_n=3):
    """Correspondence set of registration_ransac_based_on_feature_matching: i -> nn(i); with the mutual filter only
    pairs that pick each other, unless fewer than 3 * ransac_n survive (then the unfiltered set)."""
    i = np.arange(len(nn_st), dtype=np.int32)
    all_c = np.stack([i, nn_st.astype(np.int32)], axis=1)
    if not mutual_filter:
        return all_c
    keep = nn_ts[nn_st] == i
    mut = all_c[keep]
    return mut if len(mut) >= ransac_n * 3 else all_c


def ransac_correspondence(src, tgt, corres, max_corr, ransac_n=3, edge_sim=0.95, dist_thr=None, max_iter=250000,
                          confidence=0.999, seed=1234):
    src, tgt = _f32(src), _f32(tgt)
    cor = np.ascontiguousarray(corres, dtype=np.int32).reshape(-1, 2)
    T = np.zeros(16, np.float64)
    fit, rmse, best, val = C.c_double(), C.c_double(), C.c_int32(), C.c_int64()
    rc = lib().kpo_ransac_correspondence(_p(src), _p(tgt), _p(cor), C.c_long(cor.shape[0]), C.c_double(max_corr), C.c_int(ransac_n),
                                         C.c_double(edge_sim), C.c_double(max_corr if dist_thr is None else dist_thr),
                                         C.c_int(max_iter), C.c_double(confidence), C.c_uint64(seed), _p(T), C.byref(fit),
                                         C.byref(rmse), C.byref(best), C.byref(val))
    if rc != 0:
        raise ValueError("oracle ransac_correspondence: bad arguments")
    return {"T": T.reshape(4, 4), "fitness": fit.value, "rmse": rmse.value, "best_iter": best.value, "validated": val.value}


# ------------------------------------------------------------ compositions --
def filter_outliers(pts, nb_neighbors=200, std_ratio=3.0, voxel_size=0.02):
    """preprocessing/filtering.py:12-25 restated on arrays: voxel -> SOR, returns kept points."""
    v = voxel_downsample(pts, voxel_size)
    keep, _, _ = sor(v["points"], nb_neighbors, std_ratio)
    return v["points"][keep.astype(bool)]


def remove_floor(pts, band=200, thr=30, ransac_n=30, iters=2000, nb_neighbors=50, std_ratio=0.30, seed=1234):
    """floor_removal.py:64-73 restated on arrays."""
    pts = _f32(pts)
    low = band_mask(pts, band).astype(bool)
    floor, upper = pts[low], pts[~low]
    plane, inl, best, _ = ransac_plane(floor, thr, ransac_n, iters, seed=seed)
    merged = np.concatenate([floor[~inl.astype(bool)], upper], axis=0)
    keep, _, _ = sor(merged, nb_neighbors, std_ratio)
    return merged[keep.astype(bool)], plane, inl


def _sor_or_all(pts, k, ratio):
    """SOR's kept rows; k = 0 switches the stage off (every row kept), as the engine's sor_k / floor_sor_k = 0 do."""
    if k <= 0:
        return pts
    keep, _, _ = sor(pts, k, ratio)
    return pts[keep.astype(bool)]


def frame_pipeline(cfg, depth_f, tab, T_fuse, T_icp, want_icp=True, timings=None, stages=False):
    """One frame of BASELINE config C4 on the CPU: the composition the batched GPU driver implements
    (preprocessing/data.py:44-61 -> floor_removal.py:64-73 -> preprocessing/registration.py:65-86).
    ``cfg`` is any object with the PipelineConfig field names.  ``timings`` (dict) collects seconds per stage.

    Every frame gets a result, by the engine's rules where upstream would raise (DESIGN §6): an empty cloud runs
    every stage as a no-op; fewer SOR survivors than ``ransac_n`` skip floor removal (the SOR output is the frame's
    cloud); a band smaller than ``ransac_n`` has no plane and no inliers (the band and the upper part still go
    through the floor SOR).  ``stages=True`` adds ``n_lo`` (band), ``n_rest`` (band outliers), ``n_merged``,
    ``n_fsor`` and, per sensor, ``nv_icp`` (valid rows of the ICP input) and ``n_icp`` (its voxel count): the
    numbers ``FramePipeline.frame_counts()`` reports (0 for a stage that does not run)."""
    import time as _t
    S, P = cfg.n_sensors, cfg.pixels
    tick = [_t.perf_counter()]

    def lap(name):
        now = _t.perf_counter()
        if timings is not None:
            timings[name] = timings.get(name, 0.0) + (now - tick[0])
        tick[0] = now

    xyz, valid, _ = unproject(depth_f[None], tab, T_fuse, flags=cfg.unproject_flags, scale=cfg.scale)
    fused = xyz[0]
    out = {"n_fused": int(valid.sum())}
    lap("unproject")
    v = voxel_downsample(fused, cfg.voxel_size)
    out["n_voxel"] = v["m"]
    lap("voxel")
    A = _sor_or_all(v["points"], cfg.sor_k, cfg.sor_ratio)
    out["n_sor"] = len(A)
    lap("sor")
    st = {"n_lo": 0, "n_rest": 0, "n_merged": 0, "n_fsor": 0}
    out["n_floor_inliers"] = 0
    out["points"] = A
    if cfg.do_floor and len(A) > 0:
        low = band_mask(A, cfg.floor_band, 1).astype(bool)
        floor, upper = A[low], A[~low]
        if len(floor) >= cfg.ransac_n:
            plane, inl, best, _ = ransac_plane(floor, cfg.ransac_thr, cfg.ransac_n, cfg.ransac_iters, seed=cfg.seed)
            inl = inl.astype(bool)
        else:                                   # no hypothesis can be drawn: no plane, nobody is an inlier
            plane, inl = np.full(4, np.nan), np.zeros(len(floor), bool)
        merged = np.concatenate([floor[~inl], upper], 0)
        lap("ransac")
        fin = _sor_or_all(merged, cfg.floor_sor_k, cfg.floor_sor_ratio)
        lap("floor_sor")
        st.update(n_lo=len(floor), n_rest=len(floor) - int(inl.sum()), n_merged=len(merged),
                  n_fsor=len(fin) if cfg.floor_sor_k > 0 else 0)
        if len(A) >= cfg.ransac_n:              # else the floor stage is skipped: the SOR output stays the frame's cloud
            out["n_floor_inliers"] = int(inl.sum())
            out["plane"] = plane
            out["points"] = fin
    out["icp"] = []
    st["nv_icp"], st["n_icp"] = [0] * S, [0] * S
    if want_icp and cfg.do_icp and S > 1:
        tgt = voxel_downsample(fused[:P], cfg.icp_voxel)["points"]
        nrm = estimate_normals(tgt, cfg.normals_radius, cfg.normals_max_nn)
        lap("icp_prep")
        for s in range(S):
            raw, ok, _ = unproject(depth_f[None, s:s + 1], tab[s:s + 1], None, flags=cfg.unproject_flags, scale=cfg.scale)
            src = voxel_downsample(raw[0], cfg.icp_voxel)["points"]
            st["nv_icp"][s], st["n_icp"][s] = int(ok.sum()), len(src)
            if s > 0:
                out["icp"].append(icp_point_to_plane(src, tgt, nrm, cfg.icp_max_corr, init=T_icp[s], max_iter=cfg.icp_max_iter))
        lap("icp")
    if stages:
        out.update(st)
    return out
