"""The frame engine's radius outlier removal (``ror_nb_points``, ``ror_radius``) against its CPU reference
(``tests/ror_oracle.py``, composed from the oracle's pieces):
typical settings, both units, radii from far below a voxel to most of the scene, the stage combinations around it,
exact ties at d = r, ICP untouched, composed with the crop and the fixed-N output, the benchmark's batch shape, both
launch paths, and the create-time refusals.

Every case holds the engine to the oracle as ``test_gpu_engine_configs`` does (its helpers, SMALL mode): the result
counts, the per-stage counts of ``frame_counts()`` (``n_ror`` included) and the final cloud exactly, ICP to that file's
bars."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from kinectpy_b200 import _cabi, synth
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig

import ror_oracle
from test_gpu_engine_configs import SMALL, check, scene, small_cfg, solo

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VOXEL = 0.04        # small_cfg's voxel (metres)


def check_ror(oracle, cfg, depth_f, tab, T, Ti):
    ref = ror_oracle.frame_pipeline(oracle, cfg, depth_f, tab, T, Ti, stages=True)
    got, counts, raw = solo(cfg, tab, T, Ti, depth_f)
    check(got, ref, cfg.n_sensors, counts, raw)
    assert counts["n_ror"] == ref["n_ror"] and got.n_sor == ref["n_sor"]
    return got, counts, ref


@pytest.fixture(scope="module")
def small():
    return scene(SMALL, 3)


def filter_input(oracle, cfg, depth_f, tab, T):
    """The radius filter's input as the oracle computes it (voxel -> SOR)."""
    xyz, _, _ = oracle.unproject(depth_f[None], tab, T, flags=cfg.unproject_flags, scale=cfg.scale)
    v = oracle.voxel_downsample(xyz[0], cfg.voxel_size)["points"]
    return v if cfg.sor_k == 0 else v[oracle.sor(v, cfg.sor_k, cfg.sor_ratio)[0].astype(bool)]


# ------------------------------------------------------------------------------------------------ settings and units
@pytest.mark.parametrize("nb,rmult", [(1, 1.5), (8, 3.0), (200, 3.0)])
def test_typical_settings(oracle, small, nb, rmult):
    depth, tab, T, Ti = small
    got, counts, ref = check_ror(oracle, small_cfg(ror_nb_points=nb, ror_radius=rmult * VOXEL), depth[0], tab, T, Ti)
    assert ref["n_ror"] <= ref["n_sor"]
    if nb < 200:
        assert 0 < ref["n_ror"] < ref["n_sor"]


@pytest.mark.parametrize("scale", [1e-3, 1.0], ids=["m", "mm"])
def test_units(oracle, scale):
    depth, tab, T, Ti = scene(SMALL, 3, unit_scale=scale)
    unit = 1.0 if scale == 1e-3 else 1000.0
    _, _, ref = check_ror(oracle, small_cfg(scale=scale, ror_nb_points=8, ror_radius=3 * VOXEL * unit), depth[0], tab, T, Ti)
    assert 0 < ref["n_ror"] < ref["n_sor"]


# ------------------------------------------------------------------------------------------------ radii
def grid_cells(oracle, cfg, depth_f, tab, T, cell):
    """Cells of the engine's grid at `cell` over the fused cloud's bounds (k_eg_setup's count before any doubling)."""
    xyz, valid, _ = oracle.unproject(depth_f[None], tab, T, flags=cfg.unproject_flags, scale=cfg.scale)
    p = xyz[0][valid[0].astype(bool)].astype(np.float64)
    ext = p.max(0) - p.min(0)
    return float(np.prod(np.floor(ext / cell) + 2.0))


def test_tiny_radius_coarsens_the_grid(oracle, small):
    """0.01 voxel: almost no point has a neighbour (voxel means may still lie that close: the oracle's count decides).
    Cells of that size over the scene are far more than the grid holds (cap_cells = 2^20 here): k_eg_setup doubles the
    cell, which keeps the search exact."""
    depth, tab, T, Ti = small
    cfg = small_cfg(ror_nb_points=1, ror_radius=0.01 * VOXEL)
    assert grid_cells(oracle, cfg, depth[0], tab, T, cfg.ror_radius * (1 + 1e-6)) > 2 ** 20
    _, _, ref = check_ror(oracle, cfg, depth[0], tab, T, Ti)
    assert ref["n_ror"] < ref["n_sor"] // 10


def test_radius_filter_that_keeps_nothing(oracle, small):
    depth, tab, T, Ti = small
    got, counts, ref = check_ror(oracle, small_cfg(ror_nb_points=100000, ror_radius=3 * VOXEL), depth[0], tab, T, Ti)
    assert ref["n_sor"] > 0 and ref["n_ror"] == 0 and got.n_out == 0 and got.n_floor_inliers == 0
    assert [counts[k] for k in ("n_lo", "n_rest", "n_merged", "n_fsor")] == [0] * 4


def test_large_radius(oracle, small):
    """A radius of 1 m (25 voxels): a handful of cells span the scene and a query walks thousands of candidates unless
    the count ends early; nb_points = 600 keeps the dense parts only."""
    depth, tab, T, Ti = small
    _, _, ref = check_ror(oracle, small_cfg(ror_nb_points=600, ror_radius=1.0), depth[0], tab, T, Ti)
    assert 0 < ref["n_ror"] < ref["n_sor"]


# ------------------------------------------------------------------------------------------------ stage combinations
def test_without_sor(oracle, small):
    depth, tab, T, Ti = small
    _, _, ref = check_ror(oracle, small_cfg(sor_k=0, ror_nb_points=8, ror_radius=3 * VOXEL), depth[0], tab, T, Ti)
    assert ref["n_sor"] == ref["n_voxel"] and 0 < ref["n_ror"] < ref["n_sor"]


def test_without_floor_removal(oracle, small):
    depth, tab, T, Ti = small
    got, _, ref = check_ror(oracle, small_cfg(do_floor=False, ror_nb_points=8, ror_radius=3 * VOXEL), depth[0], tab, T, Ti)
    assert got.n_out == ref["n_ror"] > 0


def test_fewer_survivors_than_ransac_n_skip_the_floor(oracle, small):
    depth, tab, T, Ti = small
    base = small_cfg(ransac_n=8, ror_nb_points=1, ror_radius=3 * VOXEL)
    counts = oracle.radius_outlier(filter_input(oracle, base, depth[0], tab, T), 1, base.ror_radius)[1]
    nb = next(int(v) for v in np.unique(counts)[::-1] if 1 <= int((counts > v).sum()) < 8)
    got, _, ref = check_ror(oracle, small_cfg(ransac_n=8, ror_nb_points=nb, ror_radius=3 * VOXEL), depth[0], tab, T, Ti)
    assert ref["n_sor"] >= 8 and 1 <= ref["n_ror"] < 8 and got.n_out == ref["n_ror"] and got.n_floor_inliers == 0


# ------------------------------------------------------------------------------------------------ exact ties
def test_exact_ties_at_the_radius(oracle):
    """Millimetres, int16 unprojection, one sensor with the identity extrinsic and an 8 mm voxel: most voxels hold one
    integer point, so many pairs lie at an integer distance.  r is the integer whose pairs at exactly d = r change the
    most counts, and nb_points one at which counting them would change the kept set."""
    from scipy.spatial import cKDTree
    depth, tab, T, Ti = scene(SMALL, 1, unit_scale=1.0)
    assert np.array_equal(T[0], np.eye(4))
    base = small_cfg(S=1, scale=1.0, voxel_size=0.008, unproject_flags=_cabi.UNPROJECT_INT16 | _cabi.UNPROJECT_DROP_ANY_ZERO)
    A = filter_input(oracle, base, depth[0], tab, T)
    assert np.mean(np.all(A == np.round(A), axis=1)) > 0.5          # mostly integer points
    best = None
    for r in range(16, 41):
        strict = oracle.radius_outlier(A, 1, float(r))[1]
        incl = oracle.radius_outlier(A, 1, float(np.sqrt(r * r + 0.5)))[1]
        n = int((incl != strict).sum())
        if best is None or n > best[0]:
            best = (n, r, strict, incl)
    _, r, strict, incl = best
    pairs = cKDTree(A.astype(np.float64)).query_pairs(r + 0.01, output_type="ndarray")
    dd = A[pairs[:, 0]].astype(np.float64) - A[pairs[:, 1]].astype(np.float64)
    d2 = (dd[:, 0] * dd[:, 0] + dd[:, 1] * dd[:, 1]) + dd[:, 2] * dd[:, 2]
    assert int((d2 == r * r).sum()) > 0
    diff = incl != strict
    nb = int(np.median(strict[diff]))
    assert ((strict > nb) != (incl > nb)).any()
    cfg = small_cfg(S=1, scale=1.0, voxel_size=0.008, unproject_flags=base.unproject_flags, ror_nb_points=nb, ror_radius=float(r))
    _, _, ref = check_ror(oracle, cfg, depth[0], tab, T, Ti)
    assert ref["n_ror"] == int((strict > nb).sum())


# ------------------------------------------------------------------------------------------------ ICP, C5
def test_icp_bit_identical_with_and_without_the_radius_filter(small):
    depth, tab, T, Ti = small
    off, c_off, _ = solo(small_cfg(), tab, T, Ti, depth[0])
    on, c_on, _ = solo(small_cfg(ror_nb_points=8, ror_radius=3 * VOXEL), tab, T, Ti, depth[0])
    assert on.n_out != off.n_out and c_on["n_ror"] > 0 and c_off["n_ror"] == 0
    assert np.array_equal(on.icp_T, off.icp_T) and np.array_equal(on.icp_iters, off.icp_iters)
    assert np.array_equal(on.icp_fitness, off.icp_fitness) and np.array_equal(on.icp_rmse, off.icp_rmse)
    assert c_on["nv_icp"] == c_off["nv_icp"] and c_on["n_icp"] == c_off["n_icp"]


def test_composes_with_crop_and_fixed_output(oracle):
    from test_gpu_engine_crop_resample import crop_scene, run_solo
    depth, rgb, tab, T, Ti = crop_scene(SMALL, 3)
    cfg = small_cfg(do_crop=True, resample_n=64, ror_nb_points=4, ror_radius=2 * VOXEL)
    ref = ror_oracle.frame_pipeline(oracle, cfg, depth[0], tab, T, Ti, stages=True, rgb_f=rgb[0], frame_id=0)
    got, counts, raw = run_solo(cfg, tab, T, Ti, depth[0], rgb[0], want_fixed=True)
    check(got, ref, 3, counts, raw)
    assert counts["n_ror"] == ref["n_ror"] and 0 < ref["n_ror"] < ref["n_sor"]
    assert ref["fixed_status"] == 0 and np.array_equal(got.fixed, ref["fixed"])


# ------------------------------------------------------------------------------------------------ batch shape
def test_bench_batch_shape(oracle):
    depth, tab, T = synth.render_sequence(synth.WFOV, 2, 3)
    Tf = synth.scale_extrinsics(T, 1e-3)
    Ti = np.stack([synth.perturbed_extrinsic(Tf[s], 0.3, (3, -3, 3), unit_scale=1e-3) if s else Tf[s] for s in range(3)])
    cfg = PipelineConfig(n_sensors=3, pixels=synth.WFOV.pixels, n_streams=16, ror_nb_points=8, ror_radius=0.03)
    refs = [ror_oracle.frame_pipeline(oracle, cfg, depth[f], tab, Tf, Ti, stages=True) for f in range(2)]
    assert all(0 < r["n_ror"] < r["n_sor"] for r in refs)
    pipe = FramePipeline(cfg, tab, Tf, Ti)
    assert pipe.frames_in_flight() == (8, 2)
    got = pipe.run(np.ascontiguousarray(depth[np.arange(16) % 2]), want_points=True)
    pipe.close()
    for f, g in enumerate(got):
        ref = refs[f % 2]
        assert (g.n_fused, g.n_voxel, g.n_sor, g.n_floor_inliers, g.n_out) == \
            (ref["n_fused"], ref["n_voxel"], ref["n_sor"], ref["n_floor_inliers"], len(ref["points"])), f
        assert np.array_equal(g.points, ref["points"]), f
        for i in range(2):
            assert np.abs(g.icp_T[i] - ref["icp"][i]["T"]).max() < 1e-4, (f, i)


# ------------------------------------------------------------------------------------------------ launch paths
# Knobs read once per process: each variant runs in a fresh interpreter.
_CHILD = r"""
import json, sys
import numpy as np
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig
a = np.load(sys.argv[1])
pipe = FramePipeline(PipelineConfig(**json.loads(sys.argv[2])), a["tab"], a["T"], a["Ti"])
g = pipe.run(a["depth"], want_points=True)
c = pipe.frame_counts()
np.savez(sys.argv[3], points=np.concatenate([x.points for x in g]), n_ror=c["n_ror"],
         res=np.array([[x.n_fused, x.n_voxel, x.n_sor, x.n_floor_inliers, x.n_out] for x in g]),
         icp=np.stack([x.icp_T for x in g]))
pipe.close()
"""


def test_launch_paths(oracle, tmp_path):
    depth, tab, T, Ti = scene(SMALL, 3, frames=(0, 1, 2))
    np.savez(tmp_path / "in.npz", depth=depth, tab=tab, T=T, Ti=Ti)
    cfg = small_cfg(n_streams=4, ror_nb_points=8, ror_radius=3 * VOXEL)
    refs = [ror_oracle.frame_pipeline(oracle, cfg, depth[f], tab, T, Ti, stages=True) for f in range(3)]
    outs = {}
    for name, env in (("graph", {}), ("direct", {"KP_PIPE_GRAPH": "0"}), ("vbi", {"KP_KNN_VBI": "1"})):
        e = dict(os.environ, **env)
        e["PYTHONPATH"] = ROOT + os.pathsep + e.get("PYTHONPATH", "")
        r = subprocess.run([sys.executable, "-c", _CHILD, str(tmp_path / "in.npz"), json.dumps(cfg.__dict__),
                            str(tmp_path / ("%s.npz" % name))], cwd=ROOT, env=e, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        outs[name] = np.load(tmp_path / ("%s.npz" % name))
    assert np.array_equal(outs["graph"]["points"], np.concatenate([r["points"] for r in refs]))
    assert outs["graph"]["res"].tolist() == [[r["n_fused"], r["n_voxel"], r["n_sor"], r["n_floor_inliers"], len(r["points"])] for r in refs]
    for name in ("direct", "vbi"):
        for k in ("points", "res", "n_ror"):
            assert np.array_equal(outs[name][k], outs["graph"][k]), (name, k)
        assert np.abs(outs[name]["icp"] - outs["graph"]["icp"]).max() < 1e-4, name


# ------------------------------------------------------------------------------------------------ refusals
@pytest.mark.parametrize("kw", [dict(ror_nb_points=-1, ror_radius=0.1), dict(ror_nb_points=1, ror_radius=0.0),
                                dict(ror_nb_points=1, ror_radius=-0.1), dict(ror_nb_points=1, ror_radius=float("nan"))],
                         ids=["nb-1", "r0", "r-neg", "r-nan"])
def test_create_refuses_bad_radius_filter(small, kw):
    _, tab, T, Ti = small
    with pytest.raises(_cabi.KinectPyB200Error) as e:
        FramePipeline(small_cfg(**kw), tab, T, Ti)
    assert e.value.code == _cabi.KP_E_ARG
