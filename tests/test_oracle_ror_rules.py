"""The CPU reference of the frame engine's radius outlier removal (``tests/ror_oracle.py``, DESIGN §6):
``radius_outlier`` filters the SOR output (the voxel output when ``sor_k = 0``) and its survivors take that cloud's place
downstream, the floor-skip test included.  Its floor stage reproduces ``oracle.frame_pipeline`` on every frame rule;
without the radius filter it is ``oracle.frame_pipeline``.  ``radius_outlier`` itself is held to a brute-force strict
count."""
import types

import numpy as np
import pytest

from kinectpy_b200 import synth
from kinectpy_b200.pipeline import PipelineConfig

import ror_oracle

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


def kept(pts, keep):
    return pts[keep.astype(bool)]


def filter_input(oracle, c, d, tab, T):
    """The radius filter's input, restated: voxel -> SOR (or the voxel output when sor_k = 0)."""
    xyz, _, _ = oracle.unproject(d[None], tab, T, flags=c.unproject_flags, scale=c.scale)
    v = oracle.voxel_downsample(xyz[0], c.voxel_size)["points"]
    return v if c.sor_k == 0 else kept(v, oracle.sor(v, c.sor_k, c.sor_ratio)[0])


def restated(oracle, c, d, tab, T):
    """voxel -> SOR -> radius outlier removal -> band -> RANSAC -> merge -> floor SOR, by hand."""
    A = filter_input(oracle, c, d, tab, T)
    R = kept(A, oracle.radius_outlier(A, c.ror_nb_points, c.ror_radius)[0])
    out = {"n_sor": len(A), "n_ror": len(R), "n_floor_inliers": 0, "points": R}
    if len(R) < c.ransac_n:
        return out
    low = oracle.band_mask(R, c.floor_band, 1).astype(bool)
    floor, upper = R[low], R[~low]
    _, inl, _, _ = oracle.ransac_plane(floor, c.ransac_thr, c.ransac_n, c.ransac_iters, seed=c.seed)
    inl = inl.astype(bool)
    merged = np.concatenate([floor[~inl], upper], 0)
    out.update(n_floor_inliers=int(inl.sum()), points=kept(merged, oracle.sor(merged, c.floor_sor_k, c.floor_sor_ratio)[0]),
               n_lo=len(floor), n_merged=len(merged))
    return out


@pytest.mark.parametrize("kw", [{}, dict(sor_k=0), dict(floor_sor_k=0), dict(do_floor=False), dict(sor_k=1),
                                dict(ransac_n=8, floor_band=0.01), dict(ransac_n=64, sor_k=1, sor_ratio=1e9)],
                         ids=["default", "sor_off", "fsor_off", "no_floor", "sor_keeps_nothing", "small_band", "raw_voxels"])
def test_floor_stage_restates_the_oracle(oracle, frame, kw):
    """ror_oracle.floor_stage on the filter output of the oracle's composition is that composition's floor stage."""
    d, tab, T, Ti = frame
    c = cfg(**kw)
    ref = oracle.frame_pipeline(c, d, tab, T, Ti, want_icp=False, stages=True)
    A = oracle.frame_pipeline(types.SimpleNamespace(**dict(vars(c), do_floor=False)), d, tab, T, Ti, want_icp=False)["points"]
    pts, ninl, st = ror_oracle.floor_stage(oracle, c, A)
    assert np.array_equal(pts, ref["points"]) and ninl == ref["n_floor_inliers"]
    assert st == {k: ref[k] for k in ("n_lo", "n_rest", "n_merged", "n_fsor")}


def test_floor_stage_of_an_empty_frame(oracle, frame):
    d, tab, T, Ti = frame
    pts, ninl, st = ror_oracle.floor_stage(oracle, cfg(), np.zeros((0, 3), np.float32))
    ref = oracle.frame_pipeline(cfg(), np.zeros_like(d), tab, T, Ti, want_icp=False, stages=True)
    assert pts.shape == ref["points"].shape == (0, 3) and ninl == 0 and list(st.values()) == [0] * 4


@pytest.mark.parametrize("sor_k", [20, 0])
@pytest.mark.parametrize("nb,rmult", [(1, 1.5), (8, 3.0)])
def test_composition_with_the_radius_filter(oracle, frame, sor_k, nb, rmult):
    """ror_oracle.frame_pipeline against the composition restated by hand; ICP is the oracle's, untouched."""
    d, tab, T, Ti = frame
    c = cfg(sor_k=sor_k, ror_nb_points=nb, ror_radius=rmult * 0.04)
    o = ror_oracle.frame_pipeline(oracle, c, d, tab, T, Ti, want_icp=False, stages=True)
    r = restated(oracle, c, d, tab, T)
    assert 0 < r["n_ror"] < r["n_sor"]                   # the filter removes some points and keeps others
    assert (o["n_sor"], o["n_ror"], o["n_floor_inliers"]) == (r["n_sor"], r["n_ror"], r["n_floor_inliers"])
    assert (o["n_lo"], o["n_merged"]) == (r["n_lo"], r["n_merged"])
    assert np.array_equal(o["points"], r["points"])


def test_floor_skip_counts_the_radius_survivors(oracle, frame):
    """nb_points chosen from the counts so that 1..ransac_n-1 points survive while the SOR keeps hundreds: the floor
    stage is skipped and the survivors are the frame's cloud."""
    d, tab, T, Ti = frame
    base = cfg(ransac_n=8, ror_nb_points=1, ror_radius=0.12)
    A = filter_input(oracle, base, d, tab, T)
    counts = oracle.radius_outlier(A, 1, 0.12)[1]
    nb = next(int(v) for v in np.unique(counts)[::-1] if 1 <= int((counts > v).sum()) < 8)
    c = cfg(ransac_n=8, ror_nb_points=nb, ror_radius=0.12)
    o = ror_oracle.frame_pipeline(oracle, c, d, tab, T, Ti, want_icp=False, stages=True)
    assert o["n_sor"] >= 8 and 1 <= o["n_ror"] < 8
    assert o["n_floor_inliers"] == 0
    assert np.array_equal(o["points"], kept(A, counts > nb))


def test_stage_off_is_the_oracles_composition(oracle, frame):
    d, tab, T, Ti = frame
    off = cfg()
    bare = types.SimpleNamespace(**{k: v for k, v in vars(off).items() if not k.startswith("ror_")})
    a = ror_oracle.frame_pipeline(oracle, off, d, tab, T, Ti, stages=True)
    b = oracle.frame_pipeline(bare, d, tab, T, Ti, stages=True)
    assert a.pop("n_ror") == 0 and a.keys() == b.keys()
    for k in a:
        if k == "icp":
            for x, y in zip(a[k], b[k]):
                assert all(np.array_equal(x[f], y[f]) for f in x)
        else:
            assert np.array_equal(a[k], b[k]), k


def test_radius_outlier_counts_strictly_on_a_lattice(oracle):
    """Integer points: d^2 is exact, so pairs at exactly d = r are decided by the strict comparison alone."""
    rng = np.random.default_rng(5)
    g = np.stack(np.meshgrid(np.arange(8), np.arange(8), np.arange(6), indexing="ij"), -1).reshape(-1, 3)
    pts = g[rng.random(len(g)) < 0.6].astype(np.float32)
    p = pts.astype(np.float64)
    diff = p[:, None, :] - p[None, :, :]
    d2 = (diff[..., 0] * diff[..., 0] + diff[..., 1] * diff[..., 1]) + diff[..., 2] * diff[..., 2]
    r = 2.0
    strict, inclusive = (d2 < r * r).sum(1), (d2 <= r * r).sum(1)
    assert (d2 == r * r).any()
    for nb in (1, 4, 8, 12):
        keep, counts = oracle.radius_outlier(pts, nb, r)
        assert np.array_equal(counts, strict)
        assert np.array_equal(keep.astype(bool), strict > nb)
    assert any(((strict > nb) != (inclusive > nb)).any() for nb in (1, 4, 8, 12))
