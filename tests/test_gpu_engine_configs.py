"""The batched frame engine (kp_pipeline_*) against the oracle's frame composition away from the default shape: 1-6
sensors, ragged and tiny pixel counts, millimetres, k at the neighbour kernels' template and size limits, knobs that
move queries between the neighbour-search levels, RANSAC ties (inside and beyond the 16 the tie pass holds) and
degenerate frames inside one batch.

Every case holds the engine to the oracle: the five result counts and the final cloud exactly, the per-stage counts of
``frame_counts()`` of a single-frame run exactly, ICP transforms within 1e-4, iterations exactly, fitness within 1e-9
and rmse within 1e-6 relative (the bars of test_gpu_parity's ICP test), and ICP slots S-1..4 of the raw result record
zero."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from kinectpy_b200 import _cabi, synth
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = synth.SensorMode("SMALL", 160, 120, 126.0, 126.0, 79.5, 59.5, "hexagon")
RAGGED = synth.SensorMode("RAGGED", 157, 113, 124.0, 124.0, 78.0, 56.0, "hexagon")     # P = 17 741: odd, no multiple of 8
TINY = synth.SensorMode("TINY", 31, 9, 24.0, 24.0, 15.0, 4.0, "hexagon")               # smaller than one K1 tile / 64 rows
# Every sub within 40 degrees of the master, where point-to-plane ICP converges on this frame (a sub at 30 degrees ends
# frame 0 after all 30 passes at fitness 0.60 in the oracle: a run that long tests conditioning, not parity).
YAWS = (0.0, 40.0, -40.0, 20.0, -20.0, 10.0)
LENGTHS = ("voxel_size", "floor_band", "ransac_thr", "icp_voxel", "icp_max_corr", "normals_radius")
STAGES = ("n_lo", "n_rest", "n_merged", "n_fsor")


def small_cfg(mode=SMALL, S=3, **kw):
    base = dict(n_sensors=S, pixels=mode.pixels, voxel_size=0.04, sor_k=20, sor_ratio=2.0, floor_band=0.25,
                ransac_thr=0.02, ransac_iters=256, floor_sor_k=20, floor_sor_ratio=1.0, icp_voxel=0.04,
                icp_max_corr=0.08, normals_radius=0.08, n_streams=1)
    base.update(kw)
    if base.get("scale", 1e-3) == 1.0:              # millimetres: every length parameter in the cloud's unit
        for k in LENGTHS:
            base[k] *= 1000.0
    return PipelineConfig(**base)


def rig(S, unit_scale=1e-3):
    """Extrinsics (master first, subs at YAWS about the person) and the perturbed ICP starts, in the cloud's unit."""
    T = np.zeros((S, 4, 4))
    for i in range(S):
        c, s = math.cos(math.radians(YAWS[i])), math.sin(math.radians(YAWS[i]))
        R = np.array([[c, 0.0, s], [0.0, 1.0, 0.0], [-s, 0.0, c]])
        T[i, :3, :3], T[i, :3, 3], T[i, 3, 3] = R, synth.PERSON_CENTRE - R @ synth.PERSON_CENTRE, 1.0
    Tu = synth.scale_extrinsics(T, unit_scale)
    Ti = np.stack([synth.perturbed_extrinsic(Tu[s], 0.3, (3, -3, 3), unit_scale=unit_scale) if s else Tu[s] for s in range(S)])
    return T, Tu, Ti


def scene(mode, S, frames=(0,), unit_scale=1e-3):
    T, Tu, Ti = rig(S, unit_scale)
    tab1 = synth.xy_table(mode)
    depth = np.stack([np.stack([synth.render_depth(mode, T[s], f, s, table=tab1) for s in range(S)]) for f in frames])
    return depth, np.repeat(tab1[None], S, axis=0).copy(), Tu, Ti


def solo(cfg, tab, T, Ti, depth_f):
    """One frame alone (one frame per launch): its output, frame_counts() and raw result record."""
    pipe = FramePipeline(cfg, tab, T, Ti)
    got = pipe.run(depth_f[None], want_points=True)[0]
    counts, raw = pipe.frame_counts(), pipe._last_raw[0]
    pipe.close()
    return got, counts, raw


def check(got, ref, S, counts=None, raw=None):
    assert (got.n_fused, got.n_voxel, got.n_sor, got.n_floor_inliers, got.n_out) == \
        (ref["n_fused"], ref["n_voxel"], ref["n_sor"], ref["n_floor_inliers"], len(ref["points"]))
    assert np.array_equal(got.points, ref["points"])
    assert len(ref["icp"]) == (S - 1 if S > 1 else 0)
    for i, r in enumerate(ref["icp"]):
        assert np.abs(got.icp_T[i] - r["T"]).max() < 1e-4, i
        assert got.icp_iters[i] == r["iters"], (i, got.icp_iters[i], r["iters"])
        assert abs(got.icp_fitness[i] - r["fitness"]) < 1e-9, (i, got.icp_fitness[i], r["fitness"])
        assert abs(got.icp_rmse[i] - r["rmse"]) <= 1e-6 * max(abs(r["rmse"]), 1e-30), (i, got.icp_rmse[i], r["rmse"])
    if counts is not None:
        assert [counts[k] for k in STAGES + ("n_out",)] == [ref[k] for k in STAGES] + [len(ref["points"])]
        assert counts["nv_icp"] == ref["nv_icp"] and counts["n_icp"] == ref["n_icp"]
    if raw is not None:
        assert raw.status == 0
        for i in range(max(S - 1, 0), 5):
            assert not any(raw.icp_T[i]) and raw.icp_fitness[i] == 0 and raw.icp_rmse[i] == 0 and raw.icp_iters[i] == 0, i


def check_solo(oracle, cfg, depth_f, tab, T, Ti):
    ref = oracle.frame_pipeline(cfg, depth_f, tab, T, Ti, stages=True)
    got, counts, raw = solo(cfg, tab, T, Ti, depth_f)
    check(got, ref, cfg.n_sensors, counts, raw)
    return got, counts, ref


# ------------------------------------------------------------------------------------------------ a. sensor counts
@pytest.fixture(scope="module")
def rigs(oracle):
    out = {}
    for S in (1, 2, 4, 6):
        depth, tab, T, Ti = scene(SMALL, S, frames=(0, 1))
        cfg = small_cfg(S=S)
        out[S] = (cfg, depth, tab, T, Ti, [oracle.frame_pipeline(cfg, depth[f], tab, T, Ti, stages=True) for f in range(2)])
    return out


@pytest.mark.parametrize("S", [1, 2, 4, 6])
def test_sensor_count_matches_oracle(rigs, S):
    cfg, depth, tab, T, Ti, refs = rigs[S]
    got, counts, raw = solo(cfg, tab, T, Ti, depth[0])
    check(got, refs[0], S, counts, raw)


def test_six_sensors_at_the_bench_batch_shape(rigs):
    """8 frames per launch of 6 sensors: 40 ICP pairs in one ICP batch."""
    cfg, depth, tab, T, Ti, refs = rigs[6]
    pipe = FramePipeline(small_cfg(S=6, n_streams=16), tab, T, Ti)
    assert pipe.frames_in_flight() == (8, 2)
    got = pipe.run(np.ascontiguousarray(depth[np.arange(16) % 2]), want_points=True)
    raws = list(pipe._last_raw)
    pipe.close()
    for f, g in enumerate(got):
        check(g, refs[f % 2], 6, raw=raws[f])


# ------------------------------------------------------------------------------------------------ b. ragged pixel counts
@pytest.mark.parametrize("scale", [1e-3, 1.0])
@pytest.mark.parametrize("flags", [3, 2])
@pytest.mark.parametrize("mode", [RAGGED, TINY], ids=["157x113", "31x9"])
def test_ragged_pixel_counts(oracle, mode, flags, scale):
    depth, tab, T, Ti = scene(mode, 3, unit_scale=scale)
    cfg = small_cfg(mode, unproject_flags=flags, scale=scale)
    got, counts, ref = check_solo(oracle, cfg, depth[0], tab, T, Ti)
    assert got.n_fused > 0



def test_ragged_frames_share_a_launch(oracle):
    """P = 17 741 with 4 frames per launch (3 frames: a short batch): the fused cloud of every frame after the first, and
    the raw ICP cloud of every sensor after the master, start off the 16-byte grid."""
    depth, tab, T, Ti = scene(RAGGED, 3, frames=(0, 1, 2))
    cfg = small_cfg(RAGGED, n_streams=4)
    pipe = FramePipeline(cfg, tab, T, Ti)
    assert pipe.frames_in_flight() == (4, 1)
    got = pipe.run(depth, want_points=True)
    raws = list(pipe._last_raw)
    pipe.close()
    for f in range(3):
        check(got[f], oracle.frame_pipeline(cfg, depth[f], tab, T, Ti), 3, raw=raws[f])

# ------------------------------------------------------------------------------------------------ c. k at the kernel limits
@pytest.fixture(scope="module")
def frame3():
    return scene(SMALL, 3)


@pytest.mark.parametrize("kw", [dict(sor_k=1), dict(sor_k=32), dict(sor_k=33), dict(sor_k=64),
                                dict(floor_sor_k=32), dict(floor_sor_k=33), dict(floor_sor_k=64),
                                dict(normals_max_nn=3), dict(normals_max_nn=64), dict(icp_max_iter=0), dict(icp_max_iter=1),
                                dict(floor_band=1e-5), dict(sor_k=0), dict(floor_sor_k=0)],
                         ids=lambda kw: "%s=%s" % next(iter(kw.items())))
def test_k_at_the_kernel_limits(oracle, frame3, kw):
    """k = 32 -> 33 switches the histogram kernel's template, 64 is its largest k; sor_k = 1 keeps nothing (every point's
    only neighbour is itself); a band of 1e-5 holds fewer points than ransac_n; 0 switches a SOR stage off."""
    depth, tab, T, Ti = frame3
    got, counts, ref = check_solo(oracle, small_cfg(**kw), depth[0], tab, T, Ti)
    if kw.get("sor_k") == 1:
        assert got.n_sor == 0 and got.n_out == 0
    if "floor_band" in kw:
        assert ref["n_lo"] < 3 and got.n_floor_inliers == 0 and ref["n_merged"] == got.n_sor


@pytest.mark.parametrize("kw", [dict(sor_k=65), dict(floor_sor_k=65), dict(normals_max_nn=65)],
                         ids=lambda kw: next(iter(kw)))
def test_k_above_the_kernel_limit_is_refused(frame3, kw):
    depth, tab, T, Ti = frame3
    with pytest.raises(_cabi.KinectPyB200Error) as e:
        FramePipeline(small_cfg(**kw), tab, T, Ti)
    assert e.value.code == _cabi.KP_E_ARG


# ------------------------------------------------------------------------------------------------ d. every search level
# Knobs read once per process (function-level statics): each variant runs in a fresh interpreter.
_CHILD = r"""
import json, sys
import numpy as np
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig
a = np.load(sys.argv[1])
pipe = FramePipeline(PipelineConfig(**json.loads(sys.argv[2])), a["tab"], a["T"], a["Ti"])
g = pipe.run(a["depth"][None], want_points=True)[0]
c = pipe.frame_counts()
np.savez(sys.argv[3], points=g.points, res=np.array([g.n_fused, g.n_voxel, g.n_sor, g.n_floor_inliers, g.n_out]),
         icp_T=g.icp_T, icp_iters=g.icp_iters, icp_fitness=g.icp_fitness, icp_rmse=g.icp_rmse,
         stages=np.array([c[k] for k in ("n_lo", "n_rest", "n_merged", "n_fsor")]), nv_icp=c["nv_icp"], n_icp=c["n_icp"],
         l0=c["leftovers_l0"], mid=c["leftovers_mid"], l1=c["leftovers_l1"])
pipe.close()
"""


def far_returns(depth_f, tab):
    """Isolated far returns in every sensor: a sparse lattice of pixels at 0.3x their depth and another at 8 m."""
    d = depth_f.copy()
    S, P = d.shape
    ok = ~np.isnan(tab[0, :, 0])
    for s in range(S):
        idx = np.flatnonzero(ok & (d[s] > 0))
        d[s, idx[(s * 37) % 211::211]] = (d[s, idx[(s * 37) % 211::211]] * 0.3).astype(np.uint16)
        d[s, idx[(s * 53 + 101) % 389::389]] = 8000
    return d


@pytest.fixture(scope="module")
def far_frame(oracle):
    depth, tab, T, Ti = scene(SMALL, 3)
    d = far_returns(depth[0], tab)
    cfg = small_cfg(sor_ratio=50.0)        # SOR keeps the isolated returns: the floor SOR searches them too
    return cfg, d, tab, T, Ti, oracle.frame_pipeline(cfg, d, tab, T, Ti, stages=True)


@pytest.mark.parametrize("env", [{}, {"KP_KNN_SLACK": "0"}, {"KP_KNN_MULT_SOR": "0.5", "KP_KNN_MULT_FSOR": "0.5"},
                                 {"KP_KNN_MID": "0"}, {"KP_KNN_L1": "hist"}, {"KP_KNN_RAD": "2"}],
                         ids=["default", "slack0", "mult0.5", "no_mid", "l1_hist", "rad2"])
def test_every_search_level_receives_queries(far_frame, env, tmp_path):
    cfg, d, tab, T, Ti, ref = far_frame
    np.savez(tmp_path / "in.npz", depth=d, tab=tab, T=T, Ti=Ti)
    e = dict(os.environ, **env)
    e["PYTHONPATH"] = ROOT + os.pathsep + e.get("PYTHONPATH", "")
    r = subprocess.run([sys.executable, "-c", _CHILD, str(tmp_path / "in.npz"), json.dumps(cfg.__dict__), str(tmp_path / "out.npz")],
                       cwd=ROOT, env=e, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    o = np.load(tmp_path / "out.npz")
    assert o["res"].tolist() == [ref["n_fused"], ref["n_voxel"], ref["n_sor"], ref["n_floor_inliers"], len(ref["points"])]
    assert np.array_equal(o["points"], ref["points"])
    assert o["stages"].tolist() == [ref[k] for k in STAGES]
    assert o["nv_icp"].tolist() == ref["nv_icp"] and o["n_icp"].tolist() == ref["n_icp"]
    for i, rr in enumerate(ref["icp"]):
        assert np.abs(o["icp_T"][i] - rr["T"]).max() < 1e-4 and o["icp_iters"][i] == rr["iters"]
        assert abs(o["icp_fitness"][i] - rr["fitness"]) < 1e-9
        assert abs(o["icp_rmse"][i] - rr["rmse"]) <= 1e-6 * rr["rmse"]
    l0, mid, l1 = o["l0"].tolist(), o["mid"].tolist(), o["l1"].tolist()
    print("leftovers %s: level 0 %s, mid %s, level 1 %s" % (env or "default", l0, mid, l1))
    if not env:
        # [0] SOR, [1] floor SOR: level 0, the mid level and level 1 each hand queries on (level 1's go to k_knn_b)
        for use in (0, 1):
            assert l0[use] > 0 and mid[use] > 0 and l1[use] > 0, (use, l0, mid, l1)
    if "KP_KNN_MID" in env:
        assert mid[:2] == [0, 0]


# ------------------------------------------------------------------------------------------------ e. RANSAC ties
# One sensor looking at a hand-built cloud (the table holds each pixel's ray): a rough floor (+-3 mm) and an exactly
# flat shelf 30 cm above it, 100 points each, and up to 300 points of clutter.  Both planes hold 100 points, so
# hypotheses of either plane tie on the best count; the shelf's have a smaller sum d^2 / sqrt(count).
NF, NCLUT = 10, 300


def tie_rig():
    r = np.random.default_rng(7)
    gx, gz = np.meshgrid(np.linspace(-1.5, 1.5, NF), np.linspace(2.0, 4.5, NF))
    floor = np.stack([gx.ravel(), 1.2 + r.uniform(-0.003, 0.003, NF * NF), gz.ravel()], 1)
    shelf = np.stack([gx.ravel() * 0.8, 0.9 + r.uniform(-0.0005, 0.0005, NF * NF), gz.ravel() * 0.9 + 0.3], 1)
    y = r.uniform(0.6, 1.12, NCLUT)
    y = np.where(np.abs(y - 0.9) < 0.05, y + 0.1, y)
    clutter = np.stack([r.uniform(-1.5, 1.5, NCLUT), y, r.uniform(2.0, 4.5, NCLUT)], 1)
    pts = np.concatenate([floor, shelf, clutter])
    z = np.rint(pts[:, 2] * 1000.0)
    tab = np.stack([pts[:, 0] / (z / 1000.0), pts[:, 1] / (z / 1000.0)], 1).astype(np.float32)
    return tab[None], z.astype(np.uint16)


def tie_frame(z, clutter, shelf=True):
    """depth uint16[1, P]: the floor, the shelf (or not) and the first `clutter` clutter points."""
    d = z.copy()
    d[2 * NF * NF + clutter:] = 0
    if not shelf:
        d[NF * NF:2 * NF * NF] = 0
    return d[None]


def ransac_ties(oracle, cfg, ref_points_band):
    """Open3D's sequential best / early-exit rule replayed over the oracle's per-hypothesis counts: the processed
    hypotheses that hold the final best count, and the oracle's winner."""
    F = ref_points_band
    _, _, best, counts = oracle.ransac_plane(F, cfg.ransac_thr, cfg.ransac_n, cfg.ransac_iters, seed=cfg.seed)
    best_fit, brk, done, ties = 0.0, float(cfg.ransac_iters), 0, []
    for h, c in enumerate(counts):
        if done > brk or c == 0:        # (count 0 = degenerate sample: skipped, not counted)
            continue
        fit = c / len(F)
        if fit > best_fit:
            best_fit, ties = fit, [h]
            brk = min(math.log(1 - 0.99999999) / math.log(1 - fit ** cfg.ransac_n), cfg.ransac_iters) if fit < 1 else 0
        elif fit == best_fit:
            ties.append(h)
        done += 1
    return ties, best


def band_of(oracle, cfg, depth_f, tab):
    xyz, _, _ = oracle.unproject(depth_f[None], tab, np.eye(4)[None], flags=cfg.unproject_flags, scale=cfg.scale)
    A = oracle.voxel_downsample(xyz[0], cfg.voxel_size)["points"]
    return A[oracle.band_mask(A, cfg.floor_band, 1).astype(bool)]


def test_ransac_ties(oracle):
    tab, z = tie_rig()
    cfg = small_cfg(S=1, pixels=z.size, voxel_size=0.01, sor_k=0, floor_band=1.0, ransac_iters=100, do_icp=False, n_streams=4)
    frames = [tie_frame(z, 40), tie_frame(z, 0), tie_frame(z, 60), tie_frame(z, 100, shelf=False)]
    ties = [ransac_ties(oracle, cfg, band_of(oracle, cfg, f, tab)) for f in frames]
    # frame 0: 11 ties, the first on the floor, the winner (a later one) on the shelf; frame 1: 24 ties, more than the
    # 16 the tie pass holds; frames 2, 3: 15 and 9 ties
    assert 2 <= len(ties[0][0]) <= 16 and ties[0][1] != ties[0][0][0], ties[0]
    assert len(ties[1][0]) > 16, ties[1]
    assert all(2 <= len(t) <= 16 for t, _ in ties[2:]), ties
    print("ties at the final best count: %s; winners %s" % ([len(t) for t, _ in ties], [(b, t[0]) for t, b in ties]))
    T = np.eye(4)[None]
    pipe = FramePipeline(cfg, tab, T)
    assert pipe.frames_in_flight() == (4, 1)
    F = len(frames)
    res = (_cabi.FrameResult * F)()
    out = pipe._ctx.empty((F, z.size, 3), np.float32)
    pipe._ctx.sync()
    depth = np.ascontiguousarray(np.stack(frames))
    rc = pipe.lib.kp_pipeline_run(pipe.handle, depth.ctypes.data, 0, F, res, out.ptr, z.size)
    assert rc == _cabi.KP_E_RANGE
    host = out.to_host()
    pipe.close()
    assert [r.status for r in res] == [0, _cabi.KP_E_RANGE, 0, 0]
    for f in (0, 2, 3):
        ref = oracle.frame_pipeline(cfg, frames[f], tab, T, T, stages=True)
        got, counts, raw = solo(small_cfg(S=1, pixels=z.size, voxel_size=0.01, sor_k=0, floor_band=1.0, ransac_iters=100,
                                          do_icp=False), tab, T, T, frames[f])
        check(got, ref, 1, counts, raw)
        r = res[f]
        assert (r.n_fused, r.n_voxel, r.n_sor, r.n_floor_inliers, r.n_out) == \
            (got.n_fused, got.n_voxel, got.n_sor, got.n_floor_inliers, got.n_out), f
        assert np.array_equal(host[f, :r.n_out], got.points), f


# ------------------------------------------------------------------------------------------------ f. degenerate frames
def test_degenerate_frames_in_one_batch(oracle):
    depth, tab, T, Ti = scene(SMALL, 3, frames=(0, 1))
    cfg = small_cfg(ransac_n=8, n_streams=16)
    zero = np.zeros_like(depth[0])
    blank_master, blank_sub = depth[0].copy(), depth[1].copy()
    blank_master[0] = 0
    blank_sub[2] = 0
    few = zero.copy()                         # 5 valid pixels: fewer than k = 20 and than ransac_n = 8
    idx = np.flatnonzero(depth[0, 0])[::997][:5]
    few[0, idx] = depth[0, 0, idx]
    two = zero.copy()                         # 2 valid pixels: SOR keeps nothing (equal mean distances, sd 0)
    two[0, idx[:2]] = depth[0, 0, idx[:2]]
    batch = np.stack([depth[0], zero, blank_master, blank_sub, few, two, depth[1], depth[0]])
    pipe = FramePipeline(cfg, tab, T, Ti)
    assert pipe.frames_in_flight() == (8, 2)
    got = pipe.run(batch, want_points=True)
    raws = list(pipe._last_raw)
    pipe.close()
    refs = [oracle.frame_pipeline(cfg, f, tab, T, Ti, stages=True) for f in batch]
    assert refs[1]["n_fused"] == 0 and refs[4]["n_sor"] == 5 and refs[5]["n_fused"] == 2 and refs[5]["n_sor"] == 0
    for f in range(8):
        check(got[f], refs[f], 3, raw=raws[f])
    solo_cfg = small_cfg(ransac_n=8)
    for f in range(8):
        g, counts, raw = solo(solo_cfg, tab, T, Ti, batch[f])
        check(g, refs[f], 3, counts, raw)
        if f in (0, 6, 7):                     # the ordinary frames: byte-identical to their solo runs
            assert np.array_equal(g.points, got[f].points) and np.array_equal(g.icp_T, got[f].icp_T)
            assert np.array_equal(g.icp_fitness, got[f].icp_fitness) and np.array_equal(g.icp_rmse, got[f].icp_rmse)
