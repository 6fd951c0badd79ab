"""The batched ICP pass with the target's neighbour lists (KP_ICP_LISTS, on by default) against the same engine with
them off: every result must be bit-identical, since the list path only decides partners the grid search would find.

Cases: the benchmark's shape (WFOV, 3 sensors, 8 frames per launch), small normals_max_nn (the k-th neighbour bounds
rho), a normals radius below the ICP gate, flying points whose normals leave level 0, an empty source and an empty
target, and 1 and 8 frames per launch.  The device tally (KP_DEBUG_ICP) must show the list deciding a share of the
points in the later passes close to what tools/icp_list_premise.py counts on the CPU (0.53-0.55 from pass 3 on)."""
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from kinectpy_b200 import synth
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = synth.SensorMode("SMALL", 160, 120, 126.0, 126.0, 79.5, 59.5, "hexagon")


def small_cfg(**kw):
    base = dict(n_sensors=3, pixels=SMALL.pixels, voxel_size=0.04, sor_k=20, sor_ratio=2.0, floor_band=0.25,
                ransac_thr=0.02, ransac_iters=256, floor_sor_k=20, floor_sor_ratio=1.0, icp_voxel=0.01,
                icp_max_corr=0.04, normals_radius=0.04, n_streams=1)
    base.update(kw)
    return PipelineConfig(**base)


def small_scene(frames=(0, 1)):
    T = np.zeros((3, 4, 4))
    for i, yaw in enumerate((0.0, 40.0, -40.0)):
        c, s = math.cos(math.radians(yaw)), math.sin(math.radians(yaw))
        R = np.array([[c, 0.0, s], [0.0, 1.0, 0.0], [-s, 0.0, c]])
        T[i, :3, :3], T[i, :3, 3], T[i, 3, 3] = R, synth.PERSON_CENTRE - R @ synth.PERSON_CENTRE, 1.0
    tab1 = synth.xy_table(SMALL)
    depth = np.stack([np.stack([synth.render_depth(SMALL, T[s], f, s, table=tab1) for s in range(3)]) for f in frames])
    Tu = synth.scale_extrinsics(T, 1e-3)
    Ti = np.stack([synth.perturbed_extrinsic(Tu[s], 0.3, (3, -3, 3)) if s else Tu[s] for s in range(3)])
    return depth, np.repeat(tab1[None], 3, axis=0).copy(), Tu, Ti


def run(monkeypatch, lists, cfg, tab, T, Ti, depth):
    monkeypatch.setenv("KP_ICP_LISTS", "1" if lists else "0")
    pipe = FramePipeline(cfg, tab, T, Ti)
    out = pipe.run(np.ascontiguousarray(depth), want_points=True)
    counts = pipe.frame_counts()
    pipe.close()
    return out, counts


def same(a, b):
    (ga, ca), (gb, cb) = a, b
    # (the neighbour searches' leftover tallies depend on the order of the points inside a grid cell, which the atomics
    # of the grid build choose run by run; every result does not)
    drop = lambda c: {k: v for k, v in c.items() if not k.startswith("leftovers")}
    assert drop(ca) == drop(cb)
    assert len(ga) == len(gb)
    for x, y in zip(ga, gb):
        assert (x.n_fused, x.n_voxel, x.n_sor, x.n_floor_inliers, x.n_out) == (y.n_fused, y.n_voxel, y.n_sor, y.n_floor_inliers, y.n_out)
        assert np.array_equal(x.icp_T, y.icp_T)
        assert np.array_equal(x.icp_fitness, y.icp_fitness) and np.array_equal(x.icp_rmse, y.icp_rmse)
        assert np.array_equal(x.icp_iters, y.icp_iters)
        assert np.array_equal(x.points, y.points)


@pytest.fixture(scope="module")
def scene2():
    return small_scene()


@pytest.mark.parametrize("kw", [dict(), dict(normals_max_nn=1), dict(normals_max_nn=2), dict(normals_max_nn=13),
                                dict(normals_radius=0.02), dict(n_streams=16)],
                         ids=["default", "max_nn1", "max_nn2", "max_nn13", "radius_below_gate", "batch8"])
def test_lists_change_nothing(monkeypatch, scene2, kw):
    depth, tab, T, Ti = scene2
    cfg = small_cfg(**kw)
    d = depth[np.arange(16 if kw.get("n_streams") else 2) % 2]
    same(run(monkeypatch, True, cfg, tab, T, Ti, d), run(monkeypatch, False, cfg, tab, T, Ti, d))


def test_flying_points(monkeypatch, scene2):
    """Isolated returns at 0.3x and at 8 m: their normals search leaves level 0, so they have no list."""
    depth, tab, T, Ti = scene2
    d = depth[:1].copy()
    ok = ~np.isnan(tab[0, :, 0])
    for s in range(3):
        idx = np.flatnonzero(ok & (d[0, s] > 0))
        d[0, s, idx[(s * 37) % 97::97]] = (d[0, s, idx[(s * 37) % 97::97]] * 0.3).astype(np.uint16)
        d[0, s, idx[(s * 53 + 11) % 389::389]] = 8000
    cfg = small_cfg(sor_ratio=50.0)
    same(run(monkeypatch, True, cfg, tab, T, Ti, d), run(monkeypatch, False, cfg, tab, T, Ti, d))


@pytest.mark.parametrize("empty", [0, 1], ids=["empty_target", "empty_source"])
def test_empty_clouds(monkeypatch, scene2, empty):
    depth, tab, T, Ti = scene2
    d = depth[:2].copy()
    d[0, empty] = 0
    cfg = small_cfg(n_streams=2)
    same(run(monkeypatch, True, cfg, tab, T, Ti, d), run(monkeypatch, False, cfg, tab, T, Ti, d))


# ------------------------------------------------------------------------------------------------ the benchmark's shape
_CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import bench
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig
mode, depth, tab, T_fuse, T_icp = bench.make_inputs("WFOV", 2, 0)
pipe = FramePipeline(PipelineConfig(n_sensors=3, pixels=mode.pixels, n_streams=16), tab, T_fuse, T_icp)
got = pipe.run(np.ascontiguousarray(depth[np.arange(8) % 2]), want_points=True)
c = pipe.frame_counts()
pipe.close()
np.savez(sys.argv[2], T=np.stack([g.icp_T for g in got]), fit=np.stack([g.icp_fitness for g in got]),
         rmse=np.stack([g.icp_rmse for g in got]), it=np.stack([g.icp_iters for g in got]),
         res=np.array([[g.n_fused, g.n_voxel, g.n_sor, g.n_floor_inliers, g.n_out] for g in got]),
         pts=np.concatenate([g.points for g in got]),
         counts=np.array(sorted((k, str(v)) for k, v in c.items() if not k.startswith("leftovers"))))
"""


def test_bench_shape_and_device_tally(tmp_path):
    out = {}
    for lists in (1, 0):
        e = dict(os.environ, KP_ICP_LISTS=str(lists), KP_DEBUG_ICP="1")
        e["PYTHONPATH"] = ROOT + os.pathsep + e.get("PYTHONPATH", "")
        f = tmp_path / ("out%d.npz" % lists)
        r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(f)], cwd=ROOT, env=e, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-4000:]
        out[lists] = (np.load(f), r.stderr)
    a, b = out[1][0], out[0][0]
    for k in ("T", "fit", "rmse", "it", "res", "pts", "counts"):
        assert np.array_equal(a[k], b[k]), k
    # tally lines: "[kp icp] pair i pass k list L grid G", summed over every run of the slot
    tally = {}
    for lists in (1, 0):
        t = np.zeros((31, 2))
        for m in re.finditer(r"\[kp icp\] pair (\d+) pass (\d+) list (\d+) grid (\d+)", out[lists][1]):
            t[int(m.group(2))] += (int(m.group(3)), int(m.group(4)))
        tally[lists] = t
    assert tally[0][:, 0].sum() == 0 and tally[0][0, 1] > 0
    on = tally[1]
    assert on[0, 0] == 0                                  # pass 0 has no previous partner
    late = on[3:][on[3:].sum(1) > 0]
    share = late[:, 0].sum() / late.sum()
    print("list share per pass:", [round(x, 3) for x in (on[:, 0] / np.maximum(on.sum(1), 1))[:16]], "passes >= 3: %.3f" % share)
    assert 0.35 < share < 0.8, share
