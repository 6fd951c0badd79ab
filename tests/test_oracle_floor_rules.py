"""The CPU reference of the frame engine's floor stage with its reported plane (``tests/floor_oracle.py``, DESIGN §6).
RANSAC mode reproduces ``oracle.frame_pipeline`` -- cloud, counts and ``plane`` -- on every frame rule; plane mode is
``oracle.plane_side`` (pcd_above_plane), which is held to a NumPy left-to-right evaluation and to the reference's own
golden case, with points lying exactly on the plane."""
import os
import types

import numpy as np
import pytest

from kinectpy_b200 import _cabi, synth
from kinectpy_b200.pipeline import PipelineConfig

import floor_oracle

MODE = synth.SensorMode("SMALL", 160, 120, 126.0, 126.0, 79.5, 59.5, "hexagon")
GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_own_arithmetic.npz"))


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


def filter_output(oracle, c, d, tab, T, Ti):
    return oracle.frame_pipeline(types.SimpleNamespace(**dict(vars(c), do_floor=False)), d, tab, T, Ti, want_icp=False)["points"]


def left_to_right(pts, a, b, c, d):
    p = np.asarray(pts, np.float32).astype(np.float64)
    return (((a * p[:, 0]) + (b * p[:, 1])) + (c * p[:, 2])) + d < 0.0


# ------------------------------------------------------------------------------------------------ RANSAC mode
RULES = [{}, dict(sor_k=0), dict(floor_sor_k=0), dict(do_floor=False), dict(sor_k=1), dict(ransac_n=8, floor_band=0.001),
         dict(ransac_n=30), dict(ransac_n=64, sor_k=1, sor_ratio=1e9)]
RULE_IDS = ["default", "sor_off", "fsor_off", "no_floor", "floor_skip", "band_below_ransac_n", "ransac_n_30", "raw_voxels"]


@pytest.mark.parametrize("kw", RULES, ids=RULE_IDS)
def test_ransac_stage_restates_the_oracle(oracle, frame, kw):
    """floor_oracle.floor_stage on the filter output is oracle.frame_pipeline's floor stage, its plane included."""
    d, tab, T, Ti = frame
    c = cfg(**kw)
    ref = oracle.frame_pipeline(c, d, tab, T, Ti, want_icp=False, stages=True)
    pts, ninl, st, plane = floor_oracle.floor_stage(oracle, c, filter_output(oracle, c, d, tab, T, Ti))
    assert np.array_equal(pts, ref["points"]) and ninl == ref["n_floor_inliers"]
    assert st == {k: ref[k] for k in ("n_lo", "n_rest", "n_merged", "n_fsor")}
    assert plane.dtype == np.float64 and plane.shape == (4,)
    assert np.array_equal(plane, ref.get("plane", np.full(4, np.nan)), equal_nan=True)


def test_ransac_rules_cover_every_plane_case(oracle, frame):
    """The rules above reach a refit plane, a skipped floor stage, a band smaller than ransac_n and no floor stage."""
    d, tab, T, Ti = frame
    planes = {}
    for kw, name in zip(RULES, RULE_IDS):
        c = cfg(**kw)
        A = filter_output(oracle, c, d, tab, T, Ti)
        _, _, st, plane = floor_oracle.floor_stage(oracle, c, A)
        planes[name] = (len(A), st["n_lo"], plane)
    assert np.isfinite(planes["default"][2]).all() and abs(np.linalg.norm(planes["default"][2][:3]) - 1) < 1e-12
    assert planes["floor_skip"][0] < 3 and np.isnan(planes["floor_skip"][2]).all()
    assert planes["band_below_ransac_n"][0] >= 8 > planes["band_below_ransac_n"][1]
    assert np.isnan(planes["band_below_ransac_n"][2]).all() and np.isnan(planes["no_floor"][2]).all()


def test_ransac_stage_of_an_empty_frame(oracle, frame):
    d, tab, T, Ti = frame
    pts, ninl, st, plane = floor_oracle.floor_stage(oracle, cfg(), np.zeros((0, 3), np.float32))
    ref = oracle.frame_pipeline(cfg(), np.zeros_like(d), tab, T, Ti, want_icp=False, stages=True)
    assert pts.shape == ref["points"].shape == (0, 3) and ninl == 0 and list(st.values()) == [0] * 4
    assert "plane" not in ref and np.isnan(plane).all()


def test_ransac_mode_is_the_oracles_composition(oracle, frame):
    d, tab, T, Ti = frame
    c = cfg()
    a = floor_oracle.frame_pipeline(oracle, c, d, tab, T, Ti, stages=True)
    b = oracle.frame_pipeline(c, d, tab, T, Ti, stages=True)
    assert np.array_equal(a.pop("floor_plane"), b.pop("plane")) and a.pop("n_ror") == 0
    assert a.keys() == b.keys()
    for k in a:
        if k == "icp":
            for x, y in zip(a[k], b[k]):
                assert all(np.array_equal(x[f], y[f]) for f in x)
        else:
            assert np.array_equal(a[k], b[k]), k


# ------------------------------------------------------------------------------------------------ plane mode
def test_plane_side_is_the_left_to_right_expression(oracle):
    rng = np.random.default_rng(3)
    pts = rng.uniform(-2, 2, (5000, 3)).astype(np.float32)
    for a, b, c, d in [(0.1, -0.9, 0.3, 0.25), tuple(rng.normal(size=4)), (0.0, 1.0, 0.0, -0.5)]:
        assert np.array_equal(oracle.plane_side(pts, a, b, c, d).astype(bool), left_to_right(pts, a, b, c, d))


def test_plane_side_drops_points_on_the_plane(oracle):
    """Lattice points and planes with integer coefficients: the expression is exact, so the rows on the plane give 0
    and the strict test drops them."""
    g = np.stack(np.meshgrid(np.arange(-4, 5), np.arange(-4, 5), np.arange(-4, 5), indexing="ij"), -1).reshape(-1, 3)
    pts = g.astype(np.float32)
    for a, b, c, d in [(0.0, 1.0, 0.0, -2.0), (1.0, 2.0, -1.0, -3.0)]:
        p = g.astype(np.float64)
        v = ((a * p[:, 0] + b * p[:, 1]) + c * p[:, 2]) + d
        keep = oracle.plane_side(pts, a, b, c, d).astype(bool)
        assert (v == 0).sum() > 0
        assert np.array_equal(keep, v < 0) and not np.array_equal(keep, v <= 0)
        assert np.array_equal(keep, left_to_right(pts, a, b, c, d))


def test_plane_side_matches_the_reference_golden_case(oracle):
    a, b, c, d = GOLD["above_plane"]
    cloud = GOLD["above_cloud"]
    keep = oracle.plane_side(cloud, a, b, c, d).astype(bool)
    assert np.array_equal(cloud[keep], GOLD["above_points"])
    assert np.array_equal(keep, left_to_right(cloud, a, b, c, d))


def test_plane_stage_composition(oracle, frame):
    """Plane mode on the filter output: plane_side, then the floor SOR, counts as kp_api.h states them."""
    d, tab, T, Ti = frame
    ref = oracle.frame_pipeline(cfg(), d, tab, T, Ti, want_icp=False)
    a, b, c, dd = ref["plane"]
    s = 1.0 if b > 0 else -1.0                          # the floor lies at the largest y: normal towards it
    pl = (s * a, s * b, s * c, s * dd + 0.02)
    c_pl = cfg(floor_mode=_cabi.FLOOR_PLANE, floor_plane=pl)
    A = filter_output(oracle, c_pl, d, tab, T, Ti)
    out = floor_oracle.frame_pipeline(oracle, c_pl, d, tab, T, Ti, want_icp=False, stages=True)
    merged = A[oracle.plane_side(A, *pl).astype(bool)]
    assert 0 < len(merged) < len(A)
    assert np.array_equal(out["points"], oracle._sor_or_all(merged, 20, 1.0))
    assert out["n_floor_inliers"] == len(A) - len(merged) and (out["n_lo"], out["n_rest"]) == (0, 0)
    assert out["n_merged"] == len(merged) and out["n_fsor"] == len(out["points"])
    assert np.array_equal(out["floor_plane"], np.array(pl))


def test_plane_that_keeps_every_row_without_floor_sor(oracle, frame):
    d, tab, T, Ti = frame
    c = cfg(floor_mode=_cabi.FLOOR_PLANE, floor_plane=(0.0, 1.0, 0.0, -1e6), floor_sor_k=0)
    A = filter_output(oracle, c, d, tab, T, Ti)
    out = floor_oracle.frame_pipeline(oracle, c, d, tab, T, Ti, want_icp=False, stages=True)
    assert len(A) > 0 and np.array_equal(out["points"], A)
    assert out["n_floor_inliers"] == 0 and out["n_merged"] == len(A) and out["n_fsor"] == 0


@pytest.mark.parametrize("d,kept", [(-1.0, True), (0.0, False), (1.0, False)])
def test_zero_normal_keeps_every_row_iff_d_is_negative(oracle, frame, d, kept):
    dep, tab, T, Ti = frame
    c = cfg(floor_mode=_cabi.FLOOR_PLANE, floor_plane=(0.0, 0.0, 0.0, d), floor_sor_k=0)
    A = filter_output(oracle, c, dep, tab, T, Ti)
    out = floor_oracle.frame_pipeline(oracle, c, dep, tab, T, Ti, want_icp=False)
    assert len(out["points"]) == (len(A) if kept else 0) and out["n_floor_inliers"] == (0 if kept else len(A))


def test_plane_mode_has_no_floor_skip(oracle, frame):
    """Two filter-output rows (fewer than ransac_n): the cut still runs."""
    A = np.array([[0.0, 0.5, 1.0], [0.0, 2.0, 1.0]], np.float32)
    c = cfg(floor_mode=_cabi.FLOOR_PLANE, floor_plane=(0.0, 1.0, 0.0, -1.0), floor_sor_k=0)
    pts, ninl, st, _ = floor_oracle.floor_stage(oracle, c, A)
    assert np.array_equal(pts, A[:1]) and ninl == 1 and st["n_merged"] == 1
    pts, ninl, st, _ = floor_oracle.floor_stage(oracle, c, A[:0])
    assert len(pts) == 0 and ninl == 0 and st["n_merged"] == 0
