"""The frame engine's floor plane: each frame's plane in its result record (RANSAC mode) and the floor cut at a
caller-given plane (``floor_mode = FLOOR_PLANE``), against the CPU reference ``tests/floor_oracle.py``.

RANSAC mode: the reported plane within 1e-9 of the oracle's refit plane (absolute on a, b, c; relative on d), NaN where
the frame has none, bit-identical run to run, and every other output unchanged.  Plane mode: the final cloud, the counts
and ``frame_counts()`` exactly, a strict cut with rows exactly on the plane, both floor SOR settings, the three-step
workflow, ICP untouched, the crop and the fixed-N output, the benchmark's batch shape, and the create-time refusals."""
import numpy as np
import pytest

from kinectpy_b200 import _cabi, synth
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig

import floor_oracle
from test_gpu_engine_configs import SMALL, check, scene, small_cfg, solo
from test_gpu_engine_crop_resample import crop_scene, run_solo

pytestmark = pytest.mark.gpu

VOXEL = 0.04        # small_cfg's voxel (metres)
PLANE = _cabi.FLOOR_PLANE


def assert_plane_close(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    if np.isnan(ref).all():
        assert np.isnan(got).all(), (got, ref)
        return
    assert np.abs(got[:3] - ref[:3]).max() <= 1e-9, (got, ref)
    assert abs(got[3] - ref[3]) <= 1e-9 * max(abs(ref[3]), 1e-300), (got, ref)


def check_floor(oracle, cfg, depth_f, tab, T, Ti, rgb_f=None, want_fixed=False):
    """One frame alone against floor_oracle: counts, frame_counts(), final cloud and ICP exactly (check()), the plane
    within 1e-9 (RANSAC mode) or bit for bit (plane mode)."""
    ref = floor_oracle.frame_pipeline(oracle, cfg, depth_f, tab, T, Ti, stages=True, rgb_f=rgb_f)
    if rgb_f is None:
        got, counts, raw = solo(cfg, tab, T, Ti, depth_f)
    else:
        got, counts, raw = run_solo(cfg, tab, T, Ti, depth_f, rgb_f, want_fixed=want_fixed)
    check(got, ref, cfg.n_sensors, counts, raw)
    assert counts["n_ror"] == ref["n_ror"]
    assert got.floor_plane.dtype == np.float64 and got.floor_plane.shape == (4,)
    if cfg.floor_mode == PLANE and cfg.do_floor:
        assert got.floor_plane.tobytes() == np.array(cfg.floor_plane, np.float64).tobytes()
    else:
        assert_plane_close(got.floor_plane, ref["floor_plane"])
    return got, counts, ref


def oriented(plane, thr):
    """The host step of the workflow: the normal turned towards the floor (the largest y), d moved by the RANSAC
    threshold so that the floor's inliers fall on the removed side."""
    a, b, c, d = (float(x) for x in plane)
    s = 1.0 if b > 0 else -1.0
    return (s * a, s * b, s * c, s * d + thr)


@pytest.fixture(scope="module")
def small():
    return scene(SMALL, 3)


@pytest.fixture(scope="module")
def small_mm():
    return scene(SMALL, 3, unit_scale=1.0)


# ------------------------------------------------------------------------------------------------ RANSAC mode: planes
@pytest.mark.parametrize("variant", ["plain", "ror", "crop"])
@pytest.mark.parametrize("scale", [1e-3, 1.0], ids=["m", "mm"])
@pytest.mark.parametrize("ransac_n", [3, 30])
def test_reported_plane(oracle, ransac_n, scale, variant):
    unit = 1.0 if scale == 1e-3 else 1000.0
    kw = dict(ransac_n=ransac_n, scale=scale)
    if variant == "ror":
        kw.update(ror_nb_points=8, ror_radius=3 * VOXEL * unit)
    if variant == "crop":
        depth, rgb, tab, T, Ti = crop_scene(SMALL, 3, unit_scale=scale)
        kw.update(do_crop=True)
        got, _, ref = check_floor(oracle, small_cfg(**kw), depth[0], tab, T, Ti, rgb_f=rgb[0])
    else:
        depth, tab, T, Ti = scene(SMALL, 3, unit_scale=scale)
        got, _, ref = check_floor(oracle, small_cfg(**kw), depth[0], tab, T, Ti)
    assert ref["n_floor_inliers"] > 0 and np.isfinite(ref["floor_plane"]).all()


def test_plane_is_bit_identical_run_to_run(small):
    depth, tab, T, Ti = small
    frames = np.ascontiguousarray(np.stack([depth[0]] * 4))
    pipe = FramePipeline(small_cfg(ransac_n=30, n_streams=4), tab, T, Ti)
    a = [g.floor_plane.tobytes() for g in pipe.run(frames)]
    b = [g.floor_plane.tobytes() for g in pipe.run(frames)]
    pipe.close()
    assert a == b and len(set(a)) == 1
    single, _, _ = solo(small_cfg(ransac_n=30), tab, T, Ti, depth[0])
    assert single.floor_plane.tobytes() == a[0]          # same plane whatever else the batch holds


def test_no_floor_stage_reports_nan(oracle, small):
    depth, tab, T, Ti = small
    got, _, _ = check_floor(oracle, small_cfg(do_floor=False), depth[0], tab, T, Ti)
    assert np.isnan(got.floor_plane).all()
    got, _, _ = check_floor(oracle, small_cfg(do_floor=False, floor_mode=PLANE, floor_plane=(0.0, 1.0, 0.0, -1.0)), depth[0], tab, T, Ti)
    assert np.isnan(got.floor_plane).all()


def test_band_smaller_than_ransac_n_reports_nan(oracle, small):
    depth, tab, T, Ti = small
    got, counts, ref = check_floor(oracle, small_cfg(ransac_n=8, floor_band=0.001), depth[0], tab, T, Ti)
    assert 0 < counts["n_lo"] < 8 and np.isnan(got.floor_plane).all()


def test_degenerate_batch_planes(oracle):
    """The 8-frame degenerate batch of test_gpu_engine_configs: an empty frame, a 5-pixel frame (floor skip), a frame whose
    SOR keeps nothing: NaN planes; the other frames' planes match the oracle, and nothing else changes."""
    depth, tab, T, Ti = scene(SMALL, 3, frames=(0, 1))
    cfg = small_cfg(ransac_n=8, n_streams=16)
    zero = np.zeros_like(depth[0])
    blank_master, blank_sub = depth[0].copy(), depth[1].copy()
    blank_master[0] = 0
    blank_sub[2] = 0
    few = zero.copy()
    idx = np.flatnonzero(depth[0, 0])[::997][:5]
    few[0, idx] = depth[0, 0, idx]
    two = zero.copy()
    two[0, idx[:2]] = depth[0, 0, idx[:2]]
    batch = np.stack([depth[0], zero, blank_master, blank_sub, few, two, depth[1], depth[0]])
    pipe = FramePipeline(cfg, tab, T, Ti)
    assert pipe.frames_in_flight() == (8, 2)
    got = pipe.run(batch, want_points=True)
    raws = list(pipe._last_raw)
    pipe.close()
    refs = [floor_oracle.frame_pipeline(oracle, cfg, f, tab, T, Ti, stages=True) for f in batch]
    for f in range(8):
        check(got[f], refs[f], 3, raw=raws[f])
        assert_plane_close(got[f].floor_plane, refs[f]["floor_plane"])
    for f in (1, 4, 5):
        assert np.isnan(got[f].floor_plane).all(), f
    for f in (0, 6, 7):
        assert np.isfinite(got[f].floor_plane).all(), f
    assert got[0].floor_plane.tobytes() == got[7].floor_plane.tobytes()


# ------------------------------------------------------------------------------------------------ plane mode
def ransac_plane_of(cfg, tab, T, Ti, depth_f):
    """Step 1 of the workflow: the engine's RANSAC-mode plane of one frame."""
    g, _, _ = solo(cfg, tab, T, Ti, depth_f)
    assert np.isfinite(g.floor_plane).all()
    return g.floor_plane


@pytest.mark.parametrize("fsor", [0, 50])
@pytest.mark.parametrize("scale", [1e-3, 1.0], ids=["m", "mm"])
def test_plane_mode_matches_reference(oracle, small, small_mm, scale, fsor):
    depth, tab, T, Ti = small if scale == 1e-3 else small_mm
    base = small_cfg(scale=scale, floor_sor_k=fsor)
    pl = oriented(ransac_plane_of(base, tab, T, Ti, depth[0]), base.ransac_thr)
    got, counts, ref = check_floor(oracle, small_cfg(scale=scale, floor_sor_k=fsor, floor_mode=PLANE, floor_plane=pl),
                                   depth[0], tab, T, Ti)
    assert 0 < ref["n_floor_inliers"] < ref["n_sor"]
    assert (counts["n_lo"], counts["n_rest"]) == (0, 0) and counts["n_merged"] == ref["n_sor"] - ref["n_floor_inliers"]
    assert counts["n_fsor"] == (len(ref["points"]) if fsor else 0)


def test_strict_cut_on_lattice_points(oracle):
    """int16 millimetres, one sensor on the identity extrinsic, an 8 mm voxel: most voxels hold one integer point, and
    the plane y = c runs through the integer row that holds the most of them.  Those rows give exactly 0 and are
    dropped; a non-strict cut would keep them."""
    depth, tab, T, Ti = scene(SMALL, 1, unit_scale=1.0)
    assert np.array_equal(T[0], np.eye(4))
    kw = dict(S=1, scale=1.0, voxel_size=0.008, sor_k=0, floor_sor_k=0,
              unproject_flags=_cabi.UNPROJECT_INT16 | _cabi.UNPROJECT_DROP_ANY_ZERO)
    A = floor_oracle.frame_pipeline(oracle, small_cfg(do_floor=False, **kw), depth[0], tab, T, Ti)["points"]
    ints = A[A[:, 1] == np.round(A[:, 1])]
    assert np.mean(np.all(A == np.round(A), axis=1)) > 0.5          # mostly integer points
    ys, n = np.unique(ints[:, 1], return_counts=True)
    y0 = float(ys[np.argmax(n)])
    assert n.max() > 10
    cfg = small_cfg(floor_mode=PLANE, floor_plane=(0.0, 1.0, 0.0, -y0), **kw)
    got, counts, ref = check_floor(oracle, cfg, depth[0], tab, T, Ti)
    assert got.n_out == int((A[:, 1] < y0).sum()) and got.n_floor_inliers == int((A[:, 1] >= y0).sum())
    assert int((A[:, 1] <= y0).sum()) > got.n_out


def test_zero_normal(oracle, small):
    depth, tab, T, Ti = small
    for d, keeps in ((-1.0, True), (0.0, False)):
        got, _, ref = check_floor(oracle, small_cfg(floor_mode=PLANE, floor_plane=(0.0, 0.0, 0.0, d), floor_sor_k=0), depth[0], tab, T, Ti)
        assert got.n_out == (got.n_sor if keeps else 0)


def test_workflow_plane_from_one_frame_for_a_batch(oracle):
    """RANSAC mode on one frame, the plane oriented on the host, then a 4-frame batch in plane mode."""
    depth, tab, T, Ti = scene(SMALL, 3, frames=(0, 1, 2, 3))
    base = small_cfg(n_streams=4)
    pl = oriented(ransac_plane_of(small_cfg(), tab, T, Ti, depth[0]), base.ransac_thr)
    cfg = small_cfg(n_streams=4, floor_mode=PLANE, floor_plane=pl)
    pipe = FramePipeline(cfg, tab, T, Ti)
    got = pipe.run(depth, want_points=True)
    raws = list(pipe._last_raw)
    pipe.close()
    for f in range(4):
        ref = floor_oracle.frame_pipeline(oracle, cfg, depth[f], tab, T, Ti, stages=True)
        check(got[f], ref, 3, raw=raws[f])
        assert 0 < ref["n_floor_inliers"] and got[f].floor_plane.tobytes() == np.array(pl).tobytes()


def test_icp_bit_identical_to_ransac_mode(small):
    depth, tab, T, Ti = small
    ran, c_ran, _ = solo(small_cfg(), tab, T, Ti, depth[0])
    pl = oriented(ran.floor_plane, 0.02)
    cut, c_cut, _ = solo(small_cfg(floor_mode=PLANE, floor_plane=pl), tab, T, Ti, depth[0])
    assert np.array_equal(cut.icp_T, ran.icp_T) and np.array_equal(cut.icp_iters, ran.icp_iters)
    assert np.array_equal(cut.icp_fitness, ran.icp_fitness) and np.array_equal(cut.icp_rmse, ran.icp_rmse)
    assert c_cut["nv_icp"] == c_ran["nv_icp"] and c_cut["n_icp"] == c_ran["n_icp"]


def test_plane_mode_composes_with_crop_and_fixed_output(oracle):
    depth, rgb, tab, T, Ti = crop_scene(SMALL, 3)
    g, _, _ = run_solo(small_cfg(do_crop=True), tab, T, Ti, depth[0], rgb[0])
    pl = oriented(g.floor_plane, 0.02)
    cfg = small_cfg(do_crop=True, resample_n=64, floor_mode=PLANE, floor_plane=pl)
    got, _, ref = check_floor(oracle, cfg, depth[0], tab, T, Ti, rgb_f=rgb[0], want_fixed=True)
    assert ref["fixed_status"] == 0 and np.array_equal(got.fixed, ref["fixed"])
    assert ref["n_floor_inliers"] > 0


def test_create_refuses_bad_floor_mode(small):
    _, tab, T, Ti = small
    for kw in (dict(floor_mode=2), dict(floor_mode=-1), dict(floor_mode=PLANE, floor_plane=(0.0, 1.0, float("nan"), 0.0)),
               dict(floor_mode=PLANE, floor_plane=(0.0, 1.0, 0.0, float("inf"))),
               dict(floor_mode=PLANE, floor_plane=(float("-inf"), 1.0, 0.0, 0.0))):
        with pytest.raises(_cabi.KinectPyB200Error) as e:
            FramePipeline(small_cfg(**kw), tab, T, Ti)
        assert e.value.code == _cabi.KP_E_ARG, kw


# ------------------------------------------------------------------------------------------------ batch shape
def test_bench_batch_shape(oracle):
    """16 WFOV frames in flight (bench.py's shape), RANSAC mode and then plane mode with the plane of frame 0."""
    depth, tab, T = synth.render_sequence(synth.WFOV, 2, 3)
    Tf = synth.scale_extrinsics(T, 1e-3)
    Ti = np.stack([synth.perturbed_extrinsic(Tf[s], 0.3, (3, -3, 3), unit_scale=1e-3) if s else Tf[s] for s in range(3)])
    frames = np.ascontiguousarray(depth[np.arange(16) % 2])
    ran_cfg = PipelineConfig(n_sensors=3, pixels=synth.WFOV.pixels, n_streams=16)
    pipe = FramePipeline(ran_cfg, tab, Tf, Ti)
    assert pipe.frames_in_flight() == (8, 2)
    ran = pipe.run(frames, want_points=True)
    pipe.close()
    pl = oriented(ran[0].floor_plane, ran_cfg.ransac_thr)
    cut_cfg = PipelineConfig(n_sensors=3, pixels=synth.WFOV.pixels, n_streams=16, floor_mode=PLANE, floor_plane=pl)
    pipe = FramePipeline(cut_cfg, tab, Tf, Ti)
    cut = pipe.run(frames, want_points=True)
    pipe.close()
    for name, cfg, got in (("ransac", ran_cfg, ran), ("plane", cut_cfg, cut)):
        refs = [floor_oracle.frame_pipeline(oracle, cfg, depth[f], tab, Tf, Ti) for f in range(2)]
        for f, g in enumerate(got):
            ref = refs[f % 2]
            assert (g.n_fused, g.n_voxel, g.n_sor, g.n_floor_inliers, g.n_out) == \
                (ref["n_fused"], ref["n_voxel"], ref["n_sor"], ref["n_floor_inliers"], len(ref["points"])), (name, f)
            assert np.array_equal(g.points, ref["points"]), (name, f)
            if name == "ransac":
                assert_plane_close(g.floor_plane, ref["floor_plane"])
            else:
                assert g.floor_plane.tobytes() == np.array(pl).tobytes()
            for i in range(2):
                assert np.abs(g.icp_T[i] - ref["icp"][i]["T"]).max() < 1e-4, (name, f, i)
        assert 0 < refs[0]["n_floor_inliers"]
