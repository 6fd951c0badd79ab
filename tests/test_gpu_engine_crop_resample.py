"""The frame engine's human crop (do_crop) and fixed-N output (resample_n) against the oracle's frame composition, with the
bars of test_gpu_engine_configs: the five counts, the per-stage counts and the final cloud exactly, ICP to 1e-4 / exact
iterations / 1e-9 fitness / 1e-6 relative rmse, and the fixed-N slot bit for bit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from kinectpy_b200 import _cabi, synth
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig

import c5_oracle
from test_gpu_engine_configs import RAGGED, SMALL, check, rig, small_cfg

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def crop_scene(mode, S, frames=(0,), unit_scale=1e-3):
    T, Tu, Ti = rig(S, unit_scale)
    tab1 = synth.xy_table(mode)
    depth = np.stack([np.stack([synth.render_depth(mode, T[s], f, s, table=tab1) for s in range(S)]) for f in frames])
    rgb = np.stack([np.stack([synth.render_segmentation(mode, T[s], f, s, table=tab1) for s in range(S)]) for f in frames])
    return depth, rgb, np.repeat(tab1[None], S, axis=0).copy(), Tu, Ti


def run_solo(cfg, tab, T, Ti, depth_f, rgb_f, want_fixed=False, frame_id=None):
    pipe = FramePipeline(cfg, tab, T, Ti)
    got = pipe.run(depth_f[None], rgb=None if rgb_f is None else rgb_f[None], want_points=True, want_fixed=want_fixed,
                   frame_ids=None if frame_id is None else [frame_id], check=False)[0]
    counts, raw = pipe.frame_counts(), pipe._last_raw[0]
    pipe.close()
    return got, counts, raw


def check_crop(oracle, cfg, depth_f, rgb_f, tab, T, Ti):
    ref = c5_oracle.frame_pipeline(oracle, cfg, depth_f, tab, T, Ti, stages=True, rgb_f=rgb_f)
    got, counts, raw = run_solo(cfg, tab, T, Ti, depth_f, rgb_f)
    check(got, ref, cfg.n_sensors, counts, raw)
    assert counts["crop_median"] == ref["crop_median"]
    assert counts["crop_median"] == [float(np.median(c5_oracle.crop_z16(depth_f[s], tab[s]))) for s in range(cfg.n_sensors)]
    return got, ref


@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("scale", [1e-3, 1.0])
@pytest.mark.parametrize("mode", [SMALL, RAGGED], ids=["even_P", "odd_P"])
def test_crop_matches_oracle(oracle, mode, scale, S):
    depth, rgb, tab, T, Ti = crop_scene(mode, S, unit_scale=scale)
    got, ref = check_crop(oracle, small_cfg(mode, S=S, scale=scale, do_crop=True), depth[0], rgb[0], tab, T, Ti)
    assert 0 < got.n_fused < int((~np.isnan(tab[:, :, 0])).sum())


def test_gate_removes_the_far_wall_patch(oracle):
    depth, rgb, tab, T, Ti = crop_scene(SMALL, 3)
    gated, _ = check_crop(oracle, small_cfg(do_crop=True), depth[0], rgb[0], tab, T, Ti)
    open_, _ = check_crop(oracle, small_cfg(do_crop=True, crop_gate=1e9), depth[0], rgb[0], tab, T, Ti)
    assert open_.n_fused > gated.n_fused


def test_depth_at_or_above_32768_moves_the_median(oracle):
    depth, rgb, tab, T, Ti = crop_scene(SMALL, 3)
    d = depth[0].copy()
    d[0, : SMALL.pixels // 2] = np.where(d[0, : SMALL.pixels // 2] > 0, 40000, 0)       # negative as int16
    got, ref = check_crop(oracle, small_cfg(do_crop=True), d, rgb[0], tab, T, Ti)
    base = float(np.median(c5_oracle.crop_z16(depth[0, 0], tab[0])))
    assert ref["crop_median"][0] < base


def test_icp_bit_identical_with_and_without_the_crop():
    depth, rgb, tab, T, Ti = crop_scene(SMALL, 3)
    off, c_off, _ = run_solo(small_cfg(), tab, T, Ti, depth[0], None)
    on, c_on, _ = run_solo(small_cfg(do_crop=True), tab, T, Ti, depth[0], rgb[0])
    assert on.n_fused < off.n_fused
    assert np.array_equal(on.icp_T, off.icp_T) and np.array_equal(on.icp_iters, off.icp_iters)
    assert np.array_equal(on.icp_fitness, off.icp_fitness) and np.array_equal(on.icp_rmse, off.icp_rmse)
    assert c_on["nv_icp"] == c_off["nv_icp"] and c_on["n_icp"] == c_off["n_icp"]


def test_rgb_required_exactly_when_cropping():
    depth, rgb, tab, T, Ti = crop_scene(SMALL, 3)
    for cfg, r in ((small_cfg(do_crop=True), None), (small_cfg(), rgb[0])):
        pipe = FramePipeline(cfg, tab, T, Ti)
        with pytest.raises(_cabi.KinectPyB200Error) as e:
            pipe.run(depth[0][None], rgb=None if r is None else r[None])
        assert e.value.code == _cabi.KP_E_ARG
        pipe.close()


@pytest.mark.parametrize("kw", [dict(resample_n=-1), dict(resample_n=16385), dict(resample_n=64, resample_mode=2)],
                         ids=["n-1", "n16385", "mode2"])
def test_create_refuses_bad_resample(kw):
    _, _, tab, T, Ti = crop_scene(SMALL, 3)
    with pytest.raises(_cabi.KinectPyB200Error) as e:
        FramePipeline(small_cfg(**kw), tab, T, Ti)
    assert e.value.code == _cabi.KP_E_ARG


def fixed_ref(lib_ctx, points, N, mode, seed, stream):
    """kp_resample_batch on one cloud (the per-op path) -> [N,3]."""
    import ctypes as C
    ctx = lib_ctx
    n = len(points)
    d = ctx.to_device(points if n else np.zeros((1, 3), np.float32), np.float32)
    out = ctx.empty((N, 3), np.float32)
    off = np.array([0, n], np.int64)
    ctx.check(ctx.lib.kp_resample_batch(ctx.handle, d.ptr, off.ctypes.data_as(C.POINTER(C.c_int64)), 1, N, mode, seed, stream,
                                        out.ptr, None))
    return out.to_host()


@pytest.mark.parametrize("case", ["random_small", "prefix_small", "random_wfov"])
def test_fixed_output_matches_oracle_and_resample_batch(oracle, case):
    if case == "random_wfov":
        # the benchmark's shape and defaults; on this synthetic room the median of a WFOV sensor is ~1.39 m (a fifth of
        # the pixels lie outside the circular FOV and count as 0), so the person at ~2.4 m needs a gate of 1.5 m
        mode, N, rmode = synth.WFOV, 4096, _cabi.RESAMPLE_RANDOM
        depth, rgb, tab, T, Ti = crop_scene(mode, 3)
        cfg = PipelineConfig(n_sensors=3, pixels=mode.pixels, do_crop=True, crop_gate=1500.0, resample_n=N, resample_mode=rmode,
                             n_streams=1)
    else:
        N, rmode = 64, (_cabi.RESAMPLE_RANDOM if case == "random_small" else _cabi.RESAMPLE_PREFIX)
        depth, rgb, tab, T, Ti = crop_scene(SMALL, 3)
        cfg = small_cfg(do_crop=True, resample_n=N, resample_mode=rmode)
    ref = c5_oracle.frame_pipeline(oracle, cfg, depth[0], tab, T, Ti, want_icp=(case != "random_wfov"), rgb_f=rgb[0], frame_id=7)
    got, _, raw = run_solo(cfg, tab, T, Ti, depth[0], rgb[0], want_fixed=True, frame_id=7)
    assert raw.status == 0 and ref["fixed_status"] == 0
    assert np.array_equal(got.points, ref["points"])
    assert np.array_equal(got.fixed, ref["fixed"])
    pipe_ctx = _cabi.default_context(0)
    assert np.array_equal(got.fixed, fixed_ref(pipe_ctx, got.points, N, rmode, cfg.seed, 7))


def test_short_frame_in_a_batch():
    depth, rgb, tab, T, Ti = crop_scene(SMALL, 3, frames=(0, 1))
    probe, _, _ = run_solo(small_cfg(do_crop=True), tab, T, Ti, depth[0], rgb[0])
    N = 64
    cfg = small_cfg(do_crop=True, resample_n=N, n_streams=16)
    few_d, few_rgb = depth[0].copy(), rgb[0].copy()
    few_rgb[:, N:] = 0                        # at most N * S crop pixels before voxel + SOR: fewer than N points remain
    few_rgb[:, : N // 4] = 0
    batch_d = np.stack([depth[0], depth[1], few_d, depth[0], depth[1], depth[0], depth[1], depth[0]])
    batch_rgb = np.stack([rgb[0], rgb[1], few_rgb, rgb[0], rgb[1], rgb[0], rgb[1], rgb[0]])
    pipe = FramePipeline(cfg, tab, T, Ti)
    assert pipe.frames_in_flight() == (8, 2)
    got = pipe.run(batch_d, rgb=batch_rgb, want_points=True, want_fixed=True, check=False)
    pipe.close()
    assert got[2].n_out < N and got[2].status == _cabi.KP_E_ARG and not got[2].fixed.any()
    for f in (0, 1, 3, 4, 5, 6, 7):
        solo, _, raw = run_solo(small_cfg(do_crop=True, resample_n=N), tab, T, Ti, batch_d[f], batch_rgb[f], want_fixed=True,
                                frame_id=f)
        assert got[f].status == 0 and raw.status == 0
        assert np.array_equal(got[f].points, solo.points) and np.array_equal(got[f].fixed, solo.fixed), f
    assert probe.n_out > N


def test_frame_ids_match_a_longer_run():
    depth, rgb, tab, T, Ti = crop_scene(SMALL, 3, frames=(0, 1, 2, 3))
    cfg = small_cfg(do_crop=True, resample_n=64, n_streams=4)
    pipe = FramePipeline(cfg, tab, T, Ti)
    full = pipe.run(depth, rgb=rgb, want_fixed=True)
    part = pipe.run(depth[[1, 3]], rgb=rgb[[1, 3]], want_fixed=True, frame_ids=[1, 3])
    dev_d, dev_rgb = pipe.upload(depth[[1, 3]], rgb[[1, 3]])
    part_dev = pipe.run(dev_d, rgb=dev_rgb, want_fixed=True, frame_ids=[1, 3])
    pipe.close()
    for i, f in enumerate((1, 3)):
        assert np.array_equal(part[i].fixed, full[f].fixed) and np.array_equal(part_dev[i].fixed, full[f].fixed)
    assert not np.array_equal(full[1].fixed, full[3].fixed)


_CHILD = r"""
import json, sys
import numpy as np
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig
a = np.load(sys.argv[1])
pipe = FramePipeline(PipelineConfig(**json.loads(sys.argv[2])), a["tab"], a["T"], a["Ti"])
g = pipe.run(a["depth"], rgb=a["rgb"], want_points=True, want_fixed=True)
np.savez(sys.argv[3], points=np.concatenate([x.points for x in g]), fixed=np.stack([x.fixed for x in g]),
         res=np.array([[x.n_fused, x.n_voxel, x.n_sor, x.n_floor_inliers, x.n_out] for x in g]),
         icp=np.stack([x.icp_T for x in g]))
pipe.close()
"""


def test_graph_replay_matches_direct_launches(tmp_path):
    depth, rgb, tab, T, Ti = crop_scene(SMALL, 3, frames=(0, 1, 2))
    np.savez(tmp_path / "in.npz", depth=depth, rgb=rgb, tab=tab, T=T, Ti=Ti)
    cfg = small_cfg(do_crop=True, resample_n=64, n_streams=4)
    outs = []
    for graph in ("1", "0"):
        e = dict(os.environ, KP_PIPE_GRAPH=graph)
        e["PYTHONPATH"] = ROOT + os.pathsep + e.get("PYTHONPATH", "")
        r = subprocess.run([sys.executable, "-c", _CHILD, str(tmp_path / "in.npz"), json.dumps(cfg.__dict__),
                            str(tmp_path / ("out%s.npz" % graph))], cwd=ROOT, env=e, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        outs.append(np.load(tmp_path / ("out%s.npz" % graph)))
    for k in ("points", "fixed", "res", "icp"):
        assert np.array_equal(outs[0][k], outs[1][k]), k
