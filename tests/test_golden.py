"""Golden vectors produced by running the REFERENCE'S OWN numpy arithmetic (tests/golden/make_golden.py,
run on a checkout of KinectPy with an open3d stand-in).
CPU part: the oracle and the host-side mirrors against the fixtures.  GPU part: the kernels, through the
reference-shaped Python surface, against the same fixtures."""
import os

import numpy as np
import pytest

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_own_arithmetic.npz"))


def test_equation_plane_matches_reference(capsys):
    from kinectpy_b200.floor_removal import equation_plane
    for tri, abcd in zip(GOLD["plane_triples"], GOLD["plane_abcd"]):
        assert np.array_equal(np.array(equation_plane(tri[0], tri[1], tri[2])), abcd)
    assert "equation of plane is" in capsys.readouterr().out      # the reference prints it (floor_removal.py:35)


def test_kalman_filter_matches_reference():
    from kinectpy_b200.preprocessing.filtering import kalman_filter
    assert np.allclose(kalman_filter(GOLD["kalman_in"]), GOLD["kalman_out"], rtol=1e-12, atol=1e-12)
    assert np.allclose(kalman_filter(GOLD["kalman_in"], ri=5, qi=2, fi=0.9, hi=1), GOLD["kalman_out_params"], rtol=1e-12, atol=1e-12)


def test_oracle_plane_side_matches_reference(oracle):
    a, b, c, d = GOLD["above_plane"]
    keep = oracle.plane_side(GOLD["above_cloud"], a, b, c, d).astype(bool)
    assert np.array_equal(GOLD["above_cloud"][keep], GOLD["above_points"])


def test_oracle_xyz16_rule_and_crop_match_reference(oracle):
    pts, valid = oracle.points_from_xyz16(GOLD["dat_xyz16"])
    assert np.array_equal(pts[valid.astype(bool)].astype(np.float64), GOLD["rgbd_points"])
    keep, med = oracle.crop_mask(GOLD["crop_filtered_img"], GOLD["dat_xyz16"], 750.0)
    assert med == float(GOLD["crop_median"])
    pts, valid = oracle.points_from_xyz16(GOLD["dat_xyz16"], keep=keep)
    assert np.array_equal(pts[valid.astype(bool)].astype(np.float64), GOLD["crop_points"])


def test_oracle_band_matches_reference(oracle):
    low = oracle.band_mask(GOLD["band_cloud"], 200, 1).astype(bool)
    assert np.array_equal(np.flatnonzero(low), GOLD["band_lower_idx"])
    assert np.array_equal(np.flatnonzero(~low), GOLD["band_upper_idx"])


def test_depth_dat_reader_matches_reference(tmp_path):
    from kinectpy_b200.utils import io as kio
    fp = str(tmp_path / "99")
    GOLD["dat_xyz16"].tofile(fp + "_depth.dat")
    assert np.array_equal(kio.load_depth(fp), GOLD["dat_xyz16"])


# ------------------------------------------------------------------ GPU ----
@pytest.mark.gpu
def test_gpu_pcd_above_plane_matches_reference():
    from kinectpy_b200 import PointCloud
    from kinectpy_b200.floor_removal import pcd_above_plane
    a, b, c, d = GOLD["above_plane"]
    out = pcd_above_plane(a, b, c, d, PointCloud(GOLD["above_cloud"]))
    assert np.array_equal(np.asarray(out.points), GOLD["above_points"])


@pytest.mark.gpu
def test_gpu_rgbd_to_pointcloud_matches_reference():
    from kinectpy_b200.utils.io import rgbd_to_pointcloud
    pcd = rgbd_to_pointcloud(GOLD["dat_rgb"], GOLD["dat_xyz16"])
    assert np.array_equal(np.asarray(pcd.points), GOLD["rgbd_points"])
    assert np.allclose(np.asarray(pcd.colors), GOLD["rgbd_colors"], atol=1e-7)      # colours are float32 on the device


@pytest.mark.gpu
def test_gpu_human_crop_matches_reference(ctx):
    import gpu_helpers as G
    from kinectpy_b200.preprocessing.data import transform_filtered_image_to_pointcloud
    keep, med = G.crop_mask(ctx, GOLD["crop_filtered_img"], GOLD["dat_xyz16"], 750.0)
    assert med == float(GOLD["crop_median"])
    pcd = transform_filtered_image_to_pointcloud(GOLD["crop_filtered_img"], GOLD["dat_xyz16"])
    assert np.array_equal(np.asarray(pcd.points), GOLD["crop_points"])
    assert np.allclose(np.asarray(pcd.colors), GOLD["crop_colors"], atol=1e-7)


@pytest.mark.gpu
def test_gpu_floor_band_matches_reference():
    from kinectpy_b200 import PointCloud
    from kinectpy_b200.floor_removal import split_floor_band
    lower, upper = split_floor_band(PointCloud(GOLD["band_cloud"]), 200)
    assert np.array_equal(np.asarray(lower.points), GOLD["band_cloud"][GOLD["band_lower_idx"]])
    assert np.array_equal(np.asarray(upper.points), GOLD["band_cloud"][GOLD["band_upper_idx"]])


# ------------------------------------------------------------------------------------------------------------------
# Wrapper-level goldens: tests/golden/reference_compositions.npz was produced by the reference's OWN wrapper functions
# (preprocessing/filtering.py, preprocessing/registration.py, the loop body of floor_removal.py) driving an `open3d`
# stand-in computed by the oracle (tests/golden/make_composition_golden.py).  They pin what the wrappers decide:
# call order, arguments and defaults, source / target roles, what is copied and returned.  The global and coloured
# registration cases are in tests/golden/reference_registrations.npz.
def _compositions(name="reference_compositions.npz"):
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name))


def _oracle_backed():
    import importlib.util
    p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_composition_golden.py")
    spec = importlib.util.spec_from_file_location("make_composition_golden", p)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_oracle_filter_outliers_composition_matches_reference_wrapper(oracle):
    g = _compositions()
    assert np.array_equal(oracle.filter_outliers(g["fo_in"], nb_neighbors=20, std_ratio=2.0, voxel_size=0.02), g["fo_out"])
    assert np.array_equal(oracle.filter_outliers(g["fo_default_in"]), g["fo_default_out"])      # 200 / 3.0 / 0.02
    assert "('voxel_down_sample', 0.02, 6060), ('remove_statistical_outlier', 200, 3.0, 6060)" in str(g["fo_default_calls"])


def test_oracle_remove_floor_composition_matches_reference_script(oracle):
    g = _compositions()
    pts, plane, inl = oracle.remove_floor(g["floor_in"])          # the script's literals are the defaults
    assert np.array_equal(pts, g["floor_out"])
    assert np.array_equal(plane, g["floor_plane"]) and np.array_equal(np.flatnonzero(inl), g["floor_inliers"])
    assert "('segment_plane', 30.0, 30, 2000," in str(g["floor_calls"]) and "('remove_statistical_outlier', 50, 0.3," in str(g["floor_calls"])


def test_mirror_wrappers_make_the_reference_wrappers_calls(oracle, monkeypatch):
    """Our Python mirrors (kinectpy_b200.preprocessing.*) run against the SAME oracle-backed stand-in the reference's
    wrappers ran against: identical results and identical call traces (the mirror skips the FPFH the reference
    computes and throws away), the input clouds untouched.  No GPU involved: this is about the wrappers' logic."""
    mod = _oracle_backed()
    PointCloud, registration, geometry = mod.oracle_backed_namespace()
    from kinectpy_b200.preprocessing import filtering as our_filtering
    from kinectpy_b200.preprocessing import registration as our_registration
    g = _compositions()
    # filter_outliers
    del mod.CALLS[:]
    src = PointCloud(g["fo_in"])
    got = our_filtering.filter_outliers(src, nb_neighbors=20, std_ratio=2.0, voxel_size=0.02)
    assert np.array_equal(np.asarray(got.points, np.float32), g["fo_out"])
    assert repr(mod.CALLS) == str(g["fo_calls"]) and np.array_equal(np.asarray(src.points, np.float32), g["fo_in"])
    del mod.CALLS[:]
    got = our_filtering.filter_outliers(PointCloud(g["fo_default_in"]))
    assert np.array_equal(np.asarray(got.points, np.float32), g["fo_default_out"]) and repr(mod.CALLS) == str(g["fo_default_calls"])
    # execute_point_to_plane_registration: sub is the ICP source, master the target (the reference's double swap)
    ns = type("G", (), {})()
    for k, v in list(vars(registration).items()) + list(vars(geometry).items()):
        setattr(ns, k, v)
    monkeypatch.setattr(our_registration, "_g", ns)
    del mod.CALLS[:]
    master, sub = PointCloud(g["reg_master"]), PointCloud(g["reg_sub"])
    T = our_registration.execute_point_to_plane_registration(master, sub, g["reg_init"], voxel_size=35)
    assert np.array_equal(np.asarray(T, np.float64), g["reg_T"])
    ref_calls = [c for c in eval(str(g["reg_calls"])) if c[0] != "compute_fpfh_feature"]
    assert mod.CALLS == ref_calls
    assert np.array_equal(np.asarray(master.points, np.float32), g["reg_master"]) and not master.has_normals()
    # and the array-level composition the frame pipeline implements (oracle pieces, same roles)
    src_d = oracle.voxel_downsample(g["reg_sub"], 35.0)["points"]
    tgt_d = oracle.voxel_downsample(g["reg_master"], 35.0)["points"]
    res = oracle.icp_point_to_plane(src_d, tgt_d, oracle.estimate_normals(tgt_d, 70.0, 40), 100.0, init=g["reg_init"], max_iter=30)
    assert np.array_equal(res["T"], g["reg_T"])


def test_mirror_fusion_and_processing_wrappers_make_the_reference_calls(oracle):
    """``fuse_and_filter`` (the frame-loop body of preprocessing/data.py:41-61) and
    ``utils.processing.statistical_outlier_removal`` (:302-310): our mirrors against the same stand-in as the
    reference's code -- master untouched, sub i transformed in place by transformation i-1, device order kept,
    filter_outliers with its defaults; same results, same calls."""
    mod = _oracle_backed()
    PointCloud, _, _ = mod.oracle_backed_namespace()
    from kinectpy_b200.preprocessing import data as our_data
    from kinectpy_b200.utils import processing as our_processing
    g = _compositions()
    clouds = [PointCloud(c) for c in g["fuse_in"]]
    del mod.CALLS[:]
    got = our_data.fuse_and_filter(clouds, list(g["fuse_T"]))
    assert np.array_equal(np.asarray(got.points, np.float32), g["fuse_out"])
    assert repr(mod.CALLS) == str(g["fuse_calls"])
    assert np.array_equal(np.asarray(clouds[0].points, np.float32), g["fuse_in"][0])          # master is not transformed
    assert not np.array_equal(np.asarray(clouds[1].points, np.float32), g["fuse_in"][1])      # subs are, in place (data.py:48)
    # the same composition on arrays (what K1 + filter_outliers compute in the frame pipeline)
    fused = np.concatenate([g["fuse_in"][0]] + [oracle.transform(g["fuse_in"][i], g["fuse_T"][i - 1]) for i in (1, 2)], axis=0)
    assert np.array_equal(oracle.filter_outliers(fused), g["fuse_out"])
    del mod.CALLS[:]
    got = our_processing.statistical_outlier_removal(PointCloud(g["so_in"]))
    assert np.array_equal(np.asarray(got.points, np.float32), g["so_out"]) and repr(mod.CALLS) == str(g["so_calls"])


def test_mirror_global_and_colored_registration_make_the_reference_calls(oracle, monkeypatch):
    """``execute_global_registration`` (registration.py:32-62) and ``execute_colored_ICP_registration`` (:89-114): our
    mirrors against the same oracle-backed stand-in as the reference's code.  Same transforms; same RANSAC / coloured-ICP
    calls with the same arguments, in the same order.  One documented difference: the reference re-runs the
    (deterministic) ``prepare_dataset`` in every RANSAC trial, the mirror runs it once."""
    mod = _oracle_backed()
    PointCloud, registration, geometry = mod.oracle_backed_namespace()
    from kinectpy_b200.preprocessing import registration as our_registration
    g = _compositions("reference_registrations.npz")
    ns = type("G", (), {})()
    for k, v in list(vars(registration).items()) + list(vars(geometry).items()):
        setattr(ns, k, v)
    monkeypatch.setattr(our_registration, "_g", ns)
    # global registration
    del mod.CALLS[:]
    registration._ransac_calls[0] = 0
    T = our_registration.execute_global_registration(PointCloud(g["glob_master"]), PointCloud(g["glob_sub"]), voxel_size=60,
                                                     ransac_n_trials=3)
    assert np.array_equal(np.asarray(T, np.float64), g["glob_T"])
    ref_calls = eval(str(g["glob_calls"]))
    is_ransac = lambda c: c[0] == "registration_ransac_based_on_feature_matching"
    assert [c for c in mod.CALLS if is_ransac(c)] == [c for c in ref_calls if is_ransac(c)] and sum(map(is_ransac, ref_calls)) == 3
    prep = [c for c in ref_calls if not is_ransac(c)]
    assert [c for c in mod.CALLS if not is_ransac(c)] == prep[:len(prep) // 3] and prep[:len(prep) // 3] * 3 == prep
    # coloured ICP: source <- master, target <- sub, every scale from the initial transform, the last scale returned
    pm, ps = PointCloud(g["col_master"]), PointCloud(g["col_sub"])
    pm.colors = g["col_colors"].astype(np.float64)
    ps.colors = g["col_colors"].astype(np.float64)
    del mod.CALLS[:]
    T = our_registration.execute_colored_ICP_registration(pm, ps, np.eye(4))
    assert np.array_equal(np.asarray(T, np.float64), g["col_T"]) and repr(mod.CALLS) == str(g["col_calls"])
