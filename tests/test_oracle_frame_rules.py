"""The oracle's frame composition (``oracle.frame_pipeline``) on frames where upstream's ``segment_plane`` would raise:
it follows the engine's rules (DESIGN §6) and returns a result for every frame the engine accepts."""
import numpy as np
import pytest

from kinectpy_b200 import synth
from kinectpy_b200.pipeline import PipelineConfig

MODE = synth.SensorMode("SMALL", 160, 120, 126.0, 126.0, 79.5, 59.5, "hexagon")


def cfg(**kw):
    base = dict(n_sensors=3, pixels=MODE.pixels, voxel_size=0.04, sor_k=20, sor_ratio=2.0, floor_band=0.25,
                ransac_thr=0.02, ransac_iters=256, floor_sor_k=20, floor_sor_ratio=1.0, icp_voxel=0.04,
                icp_max_corr=0.08, normals_radius=0.08, n_streams=1)
    base.update(kw)
    return PipelineConfig(**base)


@pytest.fixture(scope="module")
def frame():
    depth, tab, T = synth.render_sequence(MODE, 1, 3)
    Ti = np.stack([synth.perturbed_extrinsic(T[s], 0.3, (3, -3, 3)) if s else T[s] for s in range(3)])
    return depth[0], tab, T, Ti


def sor_kept(oracle, pts, k, ratio):
    keep, _, _ = oracle.sor(pts, k, ratio)
    return pts[keep.astype(bool)]


def assert_no_correspondences(r, T0):
    assert (r["iters"], r["fitness"], r["rmse"], r["ncorr"]) == (1, 0.0, 0.0, 0)
    assert np.array_equal(r["T"], T0)


def test_empty_frame(oracle, frame):
    d, tab, T, Ti = frame
    o = oracle.frame_pipeline(cfg(), np.zeros_like(d), tab, T, Ti, stages=True)
    assert [o[k] for k in ("n_fused", "n_voxel", "n_sor", "n_floor_inliers", "n_lo", "n_rest", "n_merged", "n_fsor")] == [0] * 8
    assert o["points"].shape == (0, 3)
    assert o["nv_icp"] == [0, 0, 0] and o["n_icp"] == [0, 0, 0]
    for s in (1, 2):
        assert_no_correspondences(o["icp"][s - 1], Ti[s])


def test_sor_that_keeps_nothing(oracle, frame):
    d, tab, T, Ti = frame
    o = oracle.frame_pipeline(cfg(sor_k=1), d, tab, T, Ti, stages=True)     # every point's one neighbour is itself
    assert o["n_voxel"] > 0 and o["n_sor"] == 0 and o["n_floor_inliers"] == 0 and o["points"].shape == (0, 3)
    assert [o[k] for k in ("n_lo", "n_rest", "n_merged", "n_fsor")] == [0] * 4
    assert len(o["icp"]) == 2 and all(r["fitness"] > 0.4 for r in o["icp"])       # the ICP branch is independent


def test_fewer_points_than_ransac_n_skip_the_floor_stage(oracle, frame):
    d, tab, T, Ti = frame
    few = np.zeros_like(d)
    idx = np.flatnonzero(d[0])[::997][:5]
    few[0, idx] = d[0, idx]
    c = cfg(ransac_n=8)
    o = oracle.frame_pipeline(c, few, tab, T, Ti, stages=True)
    v = oracle.voxel_downsample(oracle.unproject(few[None], tab, T, flags=3)[0][0], c.voxel_size)["points"]
    A = sor_kept(oracle, v, c.sor_k, c.sor_ratio)
    assert o["n_fused"] == 5 and 0 < o["n_sor"] < c.ransac_n and o["n_floor_inliers"] == 0
    assert np.array_equal(o["points"], A)
    # the band, RANSAC and floor SOR still run (their counts are reported) but do not decide the frame's cloud
    assert o["n_lo"] >= 1 and o["n_rest"] == o["n_lo"] and o["n_merged"] == o["n_sor"]
    assert o["nv_icp"] == [5, 0, 0] and o["n_icp"][1:] == [0, 0]
    for s in (1, 2):
        assert_no_correspondences(o["icp"][s - 1], Ti[s])


def test_band_smaller_than_ransac_n_has_no_plane(oracle, frame):
    d, tab, T, Ti = frame
    c = cfg(floor_band=1e-5)
    o = oracle.frame_pipeline(c, d, tab, T, Ti, stages=True)
    A = sor_kept(oracle, oracle.voxel_downsample(oracle.unproject(d[None], tab, T, flags=3)[0][0], c.voxel_size)["points"],
                 c.sor_k, c.sor_ratio)
    low = oracle.band_mask(A, c.floor_band, 1).astype(bool)
    assert 1 <= low.sum() < c.ransac_n and o["n_sor"] >= c.ransac_n
    merged = np.concatenate([A[low], A[~low]])
    assert o["n_floor_inliers"] == 0 and np.isnan(o["plane"]).all()
    assert (o["n_lo"], o["n_rest"], o["n_merged"]) == (low.sum(), low.sum(), len(A))
    assert np.array_equal(o["points"], sor_kept(oracle, merged, c.floor_sor_k, c.floor_sor_ratio))
    assert o["n_fsor"] == len(o["points"])


@pytest.mark.parametrize("blank", [0, 2])
def test_blank_sensor(oracle, frame, blank):
    d, tab, T, Ti = frame
    b = d.copy()
    b[blank] = 0
    o = oracle.frame_pipeline(cfg(), b, tab, T, Ti, stages=True)
    full = oracle.frame_pipeline(cfg(), d, tab, T, Ti)
    assert 0 < o["n_fused"] < full["n_fused"] and o["nv_icp"][blank] == 0 and o["n_icp"][blank] == 0
    for s in (1, 2):
        if blank in (0, s):                     # no target, or no source: one pass without correspondences
            assert_no_correspondences(o["icp"][s - 1], Ti[s])
        else:
            assert o["icp"][s - 1]["iters"] == full["icp"][s - 1]["iters"] and o["icp"][s - 1]["fitness"] > 0.4


def test_stage_switches(oracle, frame):
    """sor_k = 0 / floor_sor_k = 0 switch the stage off, as in the engine."""
    d, tab, T, Ti = frame
    o = oracle.frame_pipeline(cfg(sor_k=0, floor_sor_k=0), d, tab, T, Ti, want_icp=False, stages=True)
    assert o["n_sor"] == o["n_voxel"] and o["n_fsor"] == 0 and len(o["points"]) == o["n_merged"]
    assert o["n_merged"] == o["n_sor"] - o["n_floor_inliers"]
