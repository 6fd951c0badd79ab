"""The CPU reference of the frame engine's cloud input (``tests/cloud_oracle.py``): in ``floor_removal.py``'s
configuration it is ``oracle.remove_floor``, with a voxel step and the SOR alone it is ``oracle.filter_outliers``, rows
whose x is NaN are dropped without changing anything else, and on a depth frame's fused cloud it is the depth
composition (``tests/floor_oracle.py``)."""
import types

import numpy as np
import pytest

from kinectpy_b200 import synth

import cloud_oracle
import floor_oracle
from cloud_oracle import cloud_cfg, cloud_pipeline


@pytest.fixture(scope="module")
def clouds(oracle):
    return cloud_oracle.fused_clouds(oracle, frames=2)


def with_nan_rows(pts, every=7):
    out = np.insert(pts, np.arange(0, len(pts), every), np.nan, axis=0)
    out[::5, 1] = np.where(np.isnan(out[::5, 0]), 3.0, out[::5, 1])     # (a row is absent when its x is NaN, whatever y holds)
    return out.astype(np.float32)


def test_floor_removal_configuration_is_remove_floor(oracle, clouds):
    for pts in clouds:
        cfg = cloud_cfg(len(pts))
        got = cloud_pipeline(oracle, cfg, pts)
        ref, plane, inl = oracle.remove_floor(pts, seed=cfg.seed)
        assert got["n_floor_inliers"] == int(inl.sum()) > 0
        assert np.array_equal(got["points"], ref) and len(ref) > 0
        assert got["floor_plane"].tobytes() == np.asarray(plane, np.float64).tobytes()
        assert (got["n_fused"], got["n_voxel"], got["n_sor"]) == (len(pts),) * 3


def test_nan_rows_are_absent(oracle, clouds):
    pts = clouds[0]
    holed = with_nan_rows(pts)
    for kw in (dict(), dict(cloud_voxel=1, sor_k=20, sor_ratio=2.0, voxel_size=20.0)):
        a = cloud_pipeline(oracle, cloud_cfg(len(holed), **kw), holed)
        b = cloud_pipeline(oracle, cloud_cfg(len(pts), **kw), pts)
        assert a["n_fused"] == len(pts)
        assert np.array_equal(a["points"], b["points"])
        assert [a[k] for k in ("n_voxel", "n_sor", "n_floor_inliers")] == [b[k] for k in ("n_voxel", "n_sor", "n_floor_inliers")]


@pytest.mark.parametrize("k", [20, 64])
def test_voxel_and_sor_are_filter_outliers(oracle, clouds, k):
    pts = clouds[1]
    cfg = cloud_cfg(len(pts), cloud_voxel=1, voxel_size=20.0, sor_k=k, sor_ratio=3.0, do_floor=False)
    got = cloud_pipeline(oracle, cfg, pts)
    ref = oracle.filter_outliers(pts, nb_neighbors=k, std_ratio=3.0, voxel_size=20.0)
    assert np.array_equal(got["points"], ref) and got["n_sor"] == len(ref) < got["n_voxel"] < len(pts)
    assert np.isnan(got["floor_plane"]).all()


@pytest.mark.parametrize("ror", [False, True])
def test_a_fused_cloud_through_the_cloud_input_is_the_depth_composition(oracle, ror):
    """The depth composition (metres) of one frame equals the cloud composition with the voxel step on that frame's fused
    cloud, NaN rows and all."""
    mode = cloud_oracle.SMALL
    depth, tab, T = synth.render_sequence(mode, 1, 3)
    kw = dict(voxel_size=0.04, sor_k=20, sor_ratio=2.0, floor_band=0.25, ransac_thr=0.02, ransac_n=8, ransac_iters=256,
              floor_sor_k=20, floor_sor_ratio=1.0)
    if ror:
        kw.update(ror_nb_points=8, ror_radius=0.12)
    dcfg = types.SimpleNamespace(**vars(cloud_cfg(3 * mode.pixels, **kw)))
    dcfg.n_sensors, dcfg.pixels, dcfg.scale, dcfg.do_icp = 3, mode.pixels, 1e-3, False
    dcfg.unproject_flags = oracle.F_INT16 | oracle.F_DROP_ANY_ZERO
    ref = floor_oracle.frame_pipeline(oracle, dcfg, depth[0], tab, T, T, want_icp=False, stages=True)
    fused = oracle.unproject(depth[0][None], tab, T, flags=dcfg.unproject_flags, scale=1e-3)[0][0]
    assert np.isnan(fused[:, 0]).any()
    got = cloud_pipeline(oracle, cloud_cfg(len(fused), cloud_voxel=1, **kw), fused)
    for key in ("n_fused", "n_voxel", "n_sor", "n_floor_inliers", "n_ror", "n_lo", "n_rest", "n_merged", "n_fsor"):
        assert got[key] == ref[key], key
    assert np.array_equal(got["points"], ref["points"]) and ref["n_floor_inliers"] > 0
    assert got["floor_plane"].tobytes() == ref["floor_plane"].tobytes()
