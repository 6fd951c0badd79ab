"""The CPU reference of the crop and fixed-N rules (``c5_oracle.frame_pipeline`` with ``do_crop`` / ``resample_n``), the
composition the frame engine is held to: the crop against a plain restatement of the reference's own steps, ICP
untouched by the crop, and the slot of a frame that is short of N points."""
import numpy as np
import pytest

from kinectpy_b200 import synth
from kinectpy_b200.pipeline import PipelineConfig

import c5_oracle

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
    rgb = np.stack([synth.render_segmentation(MODE, T[s], 0, s, table=tab[s]) for s in range(3)])
    return depth[0], rgb, tab, T, Ti


def reference_crop(oracle, depth_f, rgb_f, tab, T, gate, scale):
    """preprocessing/data.py:165-178 on each sensor's `_depth.dat` (k4a int16 xyz), then rgbd_to_pointcloud
    (utils/io.py:29-41: the any-zero rule) and the extrinsic, written out step by step."""
    out = []
    for s in range(depth_f.shape[0]):
        _, _, xyz16 = oracle.unproject(depth_f[None, s:s + 1], tab[s:s + 1], None, flags=oracle.F_INT16, scale=1.0,
                                       want_xyz16=True)
        xyz16 = xyz16[0]
        z = xyz16[:, 2]
        median = np.median(z)
        rgb = rgb_f[s].reshape(-1, 3)
        valid_pixels = (rgb[:, 0] != 0) & (rgb[:, 1] != 0) & (rgb[:, 2] != 0)
        valid_depths = (z <= median + gate) | (z <= median - gate)
        pts, ok = oracle.points_from_xyz16(xyz16[valid_pixels & valid_depths], T[s], oracle.F_DROP_ANY_ZERO, scale)
        out.append(pts[ok.astype(bool)])
    return np.concatenate(out)


@pytest.mark.parametrize("scale", [1e-3, 1.0])
def test_crop_is_the_reference_crop(oracle, frame, scale):
    d, rgb, tab, T, Ti = frame
    Tu = synth.scale_extrinsics(T, scale)
    c = cfg(do_crop=True, scale=scale, voxel_size=0.04 if scale != 1.0 else 40.0)
    o = c5_oracle.frame_pipeline(oracle, c, d, tab, Tu, Tu, want_icp=False, rgb_f=rgb)
    ref = reference_crop(oracle, d, rgb, tab, Tu, 750.0, scale)
    assert o["n_fused"] == len(ref) > 0
    xyz, _, _ = oracle.unproject(d[None], tab, Tu, flags=c.unproject_flags, scale=scale)
    keep, meds = c5_oracle.frame_crop(oracle, rgb, d, tab, 750.0)
    assert np.array_equal(xyz[0][keep & ~np.isnan(xyz[0][:, 0])], ref)
    assert meds == [float(np.median(c5_oracle.crop_z16(d[s], tab[s]))) for s in range(3)]
    # the gate is not vacuous on this frame: the false-positive patch on the far wall survives without it
    no_gate = c5_oracle.frame_pipeline(oracle, cfg(do_crop=True, crop_gate=1e9, scale=scale, voxel_size=c.voxel_size), d, tab, Tu, Tu,
                                    want_icp=False, rgb_f=rgb)
    assert no_gate["n_fused"] > o["n_fused"]


def test_depth_at_or_above_32768_is_negative_z(oracle, frame):
    d, rgb, tab, T, Ti = frame
    big = d.copy()
    big[0, : MODE.pixels // 2] = 40000
    z = c5_oracle.crop_z16(big[0], tab[0])
    inside = ~np.isnan(tab[0, : MODE.pixels // 2, 0])
    assert (z[: MODE.pixels // 2][inside] == 40000 - 65536).all()
    _, meds = c5_oracle.frame_crop(oracle, rgb, big, tab, 750.0)
    assert meds[0] == float(np.median(z)) and meds[0] != float(np.median(c5_oracle.crop_z16(d[0], tab[0])))


def test_icp_unchanged_by_the_crop(oracle, frame):
    d, rgb, tab, T, Ti = frame
    off = c5_oracle.frame_pipeline(oracle, cfg(), d, tab, T, Ti, stages=True)
    on = c5_oracle.frame_pipeline(oracle, cfg(do_crop=True), d, tab, T, Ti, stages=True, rgb_f=rgb)
    assert on["n_fused"] < off["n_fused"]
    assert on["nv_icp"] == off["nv_icp"] and on["n_icp"] == off["n_icp"]
    for a, b in zip(on["icp"], off["icp"]):
        assert np.array_equal(a["T"], b["T"]) and a["iters"] == b["iters"]
        assert a["fitness"] == b["fitness"] and a["rmse"] == b["rmse"]


def test_short_cloud_rule(oracle):
    pts = np.arange(30, dtype=np.float32).reshape(10, 3)
    slot, status = c5_oracle.fixed_slot(oracle, pts, 16, 0, 1234, 5)
    assert status == -1 and not slot.any() and slot.shape == (16, 3)
    slot, status = c5_oracle.fixed_slot(oracle, pts, 16, 1, 1234, 5)
    assert status == 0 and np.array_equal(slot[:10], pts) and not slot[10:].any()
    slot, status = c5_oracle.fixed_slot(oracle, pts, 4, 0, 1234, 5)
    ref, _ = oracle.resample_fixed_n(pts, 4, "random", seed=1234, stream=5)
    assert status == 0 and np.array_equal(slot, ref)
    assert not np.array_equal(slot, c5_oracle.fixed_slot(oracle, pts, 4, 0, 1234, 6)[0])       # the frame id is the stream


def test_frame_pipeline_fixed_output(oracle, frame):
    d, rgb, tab, T, Ti = frame
    o = c5_oracle.frame_pipeline(oracle, cfg(do_crop=True, resample_n=64), d, tab, T, Ti, want_icp=False, rgb_f=rgb, frame_id=3)
    assert o["fixed_status"] == 0
    assert np.array_equal(o["fixed"], oracle.resample_fixed_n(o["points"], 64, seed=1234, stream=3)[0])
    o = c5_oracle.frame_pipeline(oracle, cfg(do_crop=True, resample_n=len(o["points"]) + 1), d, tab, T, Ti, want_icp=False, rgb_f=rgb)
    assert o["fixed_status"] == -1 and not o["fixed"].any()
