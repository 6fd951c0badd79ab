"""The frame engine's cloud input (``input_mode = INPUT_CLOUDS``, ``kp_pipeline_run_clouds``) against the CPU reference
``tests/cloud_oracle.py``: the five counts and the final cloud exactly, the floor plane within 1e-9, the fixed-N slot
exactly.  Also: a ragged batch whose every frame equals the frame run alone, host and device input, a cross-check with
the depth path that needs no oracle, ``remove_floor_batch`` against the per-cloud ``remove_floor``, and the refusals."""
import ctypes as C

import numpy as np
import pytest

from kinectpy_b200 import _cabi
from kinectpy_b200.floor_removal import remove_floor, remove_floor_batch
from kinectpy_b200.geometry import PointCloud
from kinectpy_b200.pipeline import FramePipeline

import cloud_oracle
from cloud_oracle import cloud_cfg, cloud_pipeline
from test_gpu_engine_configs import SMALL, scene, small_cfg

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def clouds(oracle):
    return cloud_oracle.fused_clouds(oracle, frames=3)


def run(cfg, clouds, **kw):
    pipe = FramePipeline(cfg)
    try:
        outs = pipe.run_clouds(clouds, want_points=True, **kw)
        return outs, [bytes(r) for r in pipe._last_raw]
    finally:
        pipe.close()


def check(got, ref):
    assert (got.n_fused, got.n_voxel, got.n_sor, got.n_floor_inliers, got.n_out) == \
        (ref["n_fused"], ref["n_voxel"], ref["n_sor"], ref["n_floor_inliers"], len(ref["points"]))
    assert np.array_equal(got.points, ref["points"])
    assert got.status == 0 and got.icp_T.size == 0
    plane, rp = got.floor_plane, ref["floor_plane"]
    if np.isnan(rp).all():
        assert np.isnan(plane).all()
    else:
        assert np.abs(plane[:3] - rp[:3]).max() <= 1e-9 and abs(plane[3] - rp[3]) <= 1e-9 * max(abs(rp[3]), 1e-300), (plane, rp)
    if "fixed" in ref:
        assert np.array_equal(got.fixed, ref["fixed"])


def test_floor_removal_configuration(oracle, clouds):
    cfg = cloud_cfg(max(len(c) for c in clouds), n_streams=4)
    outs, raw = run(cfg, clouds)
    for got, pts in zip(outs, clouds):
        ref = cloud_pipeline(oracle, cfg, pts)
        assert ref["n_floor_inliers"] > 0
        check(got, ref)
    # the ICP fields of the records are zero
    for r in raw:
        rec = _cabi.FrameResult.from_buffer_copy(r)
        assert not any(rec.icp_T[i][e] for i in range(5) for e in range(16)) and not any(rec.icp_iters)


@pytest.mark.parametrize("resample", [_cabi.RESAMPLE_RANDOM, _cabi.RESAMPLE_PREFIX], ids=["random", "prefix"])
@pytest.mark.parametrize("floor_mode", [_cabi.FLOOR_RANSAC, _cabi.FLOOR_PLANE], ids=["ransac", "plane"])
def test_voxel_sor_ror_floor_fixed(oracle, clouds, floor_mode, resample):
    ymax = float(np.max(clouds[0][:, 1]))
    cfg = cloud_cfg(max(len(c) for c in clouds), cloud_voxel=1, voxel_size=20.0, sor_k=20, sor_ratio=2.0, ror_nb_points=6,
                    ror_radius=60.0, floor_mode=floor_mode, floor_plane=(0.0, 1.0, 0.0, -(ymax - 120.0)), ransac_n=3,
                    ransac_iters=500, floor_sor_k=20, floor_sor_ratio=1.0, resample_n=256, resample_mode=resample, n_streams=4)
    outs, _ = run(cfg, clouds, want_fixed=True)
    for f, (got, pts) in enumerate(zip(outs, clouds)):
        ref = cloud_pipeline(oracle, cfg, pts, frame_id=f)
        assert ref["n_voxel"] < ref["n_fused"] and 0 < ref["n_ror"] < ref["n_sor"] < ref["n_voxel"] and ref["n_floor_inliers"] > 0
        check(got, ref)


def ragged_batch(clouds):
    """11 clouds: an empty one, one of exactly P rows, one with NaN rows, one whose band holds fewer than ransac_n points,
    and the saved clouds."""
    a, b, c = clouds
    holed = np.insert(b, np.arange(0, len(b), 5), np.nan, axis=0).astype(np.float32)
    P = len(holed) + 3
    exact = np.concatenate([a, c])[:P]
    assert len(exact) == P
    low = c[c[:, 1] < np.max(c[:, 1]) - 600.0]
    few = np.concatenate([low, c[:10] * np.float32(1.0) + np.array([0, np.max(c[:, 1]) - np.min(c[:10, 1]) + 500.0, 0], np.float32)])
    batch = [np.zeros((0, 3), np.float32), exact, holed, few, a, b, c, a[: 200], c, b, a]
    return batch, P


def test_ragged_batch_equals_each_frame_alone(oracle, clouds):
    batch, P = ragged_batch(clouds)
    cfg = cloud_cfg(P, n_streams=16)
    pipe = FramePipeline(cfg)
    assert pipe.frames_in_flight() == (8, 2) and len(batch) % 8
    outs = pipe.run_clouds(batch, want_points=True)
    raw = [bytes(r) for r in pipe._last_raw]
    pipe.close()
    for f, pts in enumerate(batch):
        ref = cloud_pipeline(oracle, cfg, pts)
        check(outs[f], ref)
        alone, araw = run(cloud_cfg(P), [pts])
        assert araw[0] == raw[f] and np.array_equal(alone[0].points, outs[f].points), f
    assert outs[0].n_out == 0 and outs[1].n_fused == P and outs[2].n_fused == len(clouds[1])
    assert np.isnan(outs[3].floor_plane).all() and 0 < outs[3].n_out and outs[3].n_floor_inliers == 0


def test_host_and_device_input_are_identical(ctx, clouds):
    batch, P = ragged_batch(clouds)
    for kw in (dict(), dict(cloud_voxel=1, voxel_size=20.0, sor_k=20)):
        cfg = cloud_cfg(P, n_streams=4, **kw)
        host, hraw = run(cfg, batch)
        # one leading row, so that every cloud starts off the 16-byte grid the host staging has
        flat = np.concatenate([np.full((1, 3), 7.0, np.float32)] + batch)
        off = np.concatenate([[1], 1 + np.cumsum([len(c) for c in batch])]).astype(np.int64)
        dev = ctx.to_device(flat, np.float32)
        got, draw = run(cfg, (dev, off))
        assert hraw == draw
        for h, d in zip(host, got):
            assert np.array_equal(h.points, d.points)


@pytest.mark.parametrize("floor_mode", [_cabi.FLOOR_RANSAC, _cabi.FLOOR_PLANE], ids=["ransac", "plane"])
def test_depth_filter_outputs_through_the_cloud_input_match_the_depth_path(floor_mode):
    """No oracle: the depth engine's filter outputs (do_floor = 0) through the cloud input (no voxel step, no SOR, floor
    on) give the depth engine's final clouds, floor planes and floor inliers, bit for bit."""
    depth, tab, T, Ti = scene(SMALL, 3, frames=(0, 1, 2))
    kw = dict(do_icp=False, ransac_n=8, n_streams=4)
    pipe = FramePipeline(small_cfg(do_floor=False, **kw), tab, T, Ti)
    filt = pipe.run(depth, want_points=True)
    pipe.close()
    ymax = float(np.max(filt[0].points[:, 1]))
    base = small_cfg(floor_mode=floor_mode, floor_plane=(0.0, 1.0, 0.0, -(ymax - 0.1)), **kw)
    pipe = FramePipeline(base, tab, T, Ti)
    full = pipe.run(depth, want_points=True)
    pipe.close()
    cfg = cloud_cfg(SMALL.pixels * 3, voxel_size=base.voxel_size, sor_k=0, floor_band=base.floor_band, ransac_thr=base.ransac_thr,
                    ransac_n=base.ransac_n, ransac_iters=base.ransac_iters, floor_sor_k=base.floor_sor_k,
                    floor_sor_ratio=base.floor_sor_ratio, floor_mode=floor_mode, floor_plane=base.floor_plane, seed=base.seed,
                    n_streams=4)
    got, _ = run(cfg, [f.points for f in filt])
    for g, d in zip(got, full):
        assert d.n_floor_inliers > 0
        assert np.array_equal(g.points, d.points)
        assert g.floor_plane.tobytes() == d.floor_plane.tobytes() and g.n_floor_inliers == d.n_floor_inliers


def test_remove_floor_batch_matches_remove_floor(clouds):
    batch = remove_floor_batch([PointCloud(c) for c in clouds[:2]])
    for got, c in zip(batch, clouds[:2]):
        assert np.array_equal(got.points, remove_floor(PointCloud(c)).points)


def refused(fn):
    with pytest.raises(_cabi.KinectPyB200Error) as e:
        fn()
    assert e.value.code == _cabi.KP_E_ARG


def test_refusals(ctx, clouds):
    P = max(len(c) for c in clouds)
    refused(lambda: FramePipeline(cloud_cfg(P, n_sensors=2)))
    refused(lambda: FramePipeline(cloud_cfg(P, do_icp=True)))
    refused(lambda: FramePipeline(cloud_cfg(P, do_crop=True)))
    refused(lambda: FramePipeline(cloud_cfg(P, cloud_voxel=2)))
    pipe = FramePipeline(cloud_cfg(P))
    n0 = pipe.launch_count()
    refused(lambda: pipe.run_clouds([np.zeros((P + 1, 3), np.float32)]))
    dev = ctx.to_device(np.concatenate(clouds), np.float32)
    refused(lambda: pipe.run_clouds((dev, np.array([0, 100, 50], np.int64))))
    refused(lambda: pipe.run(np.zeros((1, 1, P), np.uint16)))
    res = (_cabi.FrameResult * 1)()
    depth, rgb = np.zeros((1, 1, P), np.uint16), np.zeros((1, 1, P, 3), np.uint8)
    assert pipe.lib.kp_pipeline_run_ex(pipe.handle, depth.ctypes.data, rgb.ctypes.data, 0, 1, None, res, None, 0, None) == _cabi.KP_E_ARG
    assert pipe.launch_count() == n0
    pipe.close()
    depth, tab, T, Ti = scene(SMALL, 1)
    dpipe = FramePipeline(small_cfg(S=1, do_icp=False), tab, T)
    n0 = dpipe.launch_count()
    refused(lambda: dpipe.run_clouds([clouds[0][:100]]))
    assert dpipe.launch_count() == n0
    dpipe.close()
