"""CUDA path vs CPU oracle on the same seeded inputs, through the C ABI (include/kp_api.h).

Bars (BASELINE.json north_star): voxel keys, kept-point masks, kNN indices and RANSAC inlier sets
bit-exact; point coordinates within 1e-5 m; converged ICP transform within 1e-4.  Because the
kernels and the oracle share one arithmetic contract (double decisions on float32 storage, fixed
operation order, canonical sums) most float outputs are compared for exact equality as well.
"""
import numpy as np
import pytest

import gpu_helpers as G
from conftest import make_surface_cloud
from kinectpy_b200 import synth

pytestmark = pytest.mark.gpu

COORD_TOL = 1e-5      # metres (north_star)
ICP_TOL = 1e-4        # rotation entries / translation (north_star)


def same_with_nan(a, b):
    return np.array_equal(a, b, equal_nan=True)


# ------------------------------------------------------------------ K1 ----
@pytest.fixture(scope="module")
def nfov2():
    depth, tab, T = synth.render_sequence(synth.NFOV, 2, 3)
    return depth, tab, T


@pytest.mark.parametrize("flags,scale", [(3, 1.0), (0, 1e-3), (2, 1e-3), (1, 1e-3)])
def test_unproject_transform_bit_exact(ctx, oracle, nfov2, flags, scale):
    depth, tab, T = nfov2
    Ts = synth.scale_extrinsics(T, scale)
    ref_xyz, ref_valid, ref16 = oracle.unproject(depth, tab, Ts, flags=flags, scale=scale, want_xyz16=bool(flags & 1))
    got = G.unproject(ctx, depth, tab, Ts, flags, scale)
    assert same_with_nan(got["xyz"], ref_xyz)
    assert np.array_equal(got["valid"], ref_valid)
    if flags & 1:
        assert np.array_equal(got["xyz16"], ref16)
    for b in range(depth.shape[0]):
        ok = ref_valid[b].astype(bool)
        assert got["nvalid"][b] == ok.sum()
        assert np.array_equal(got["bounds"][b, :3], ref_xyz[b][ok].min(0))
        assert np.array_equal(got["bounds"][b, 3:], ref_xyz[b][ok].max(0))
    # against a float64 evaluation of the same formula: the north-star coordinate tolerance
    if not (flags & 1):
        P = tab.shape[1]
        z = depth[0, 1].astype(np.float64)
        pts = np.stack([tab[1, :, 0].astype(np.float64) * z, tab[1, :, 1].astype(np.float64) * z, z], 1) * scale
        exp = pts @ Ts[1, :3, :3].T + Ts[1, :3, 3]
        ok = ref_valid[0, P:2 * P].astype(bool)
        assert np.abs(got["xyz"][0, P:2 * P][ok] - exp[ok]).max() < COORD_TOL * (scale / 1e-3)


def test_unproject_ragged_sizes(ctx, oracle):
    """P not a multiple of the tile / vector width, identity extrinsics, single sensor."""
    r = np.random.default_rng(0)
    for P in (1, 7, 1001, 2048 + 3):
        depth = r.integers(0, 6000, (2, 1, P)).astype(np.uint16)
        depth[:, :, ::5] = 0
        tab = r.uniform(-1, 1, (1, P, 2)).astype(np.float32)
        tab[0, ::11] = np.nan
        for flags in (0, 3):
            ref_xyz, ref_valid, _ = oracle.unproject(depth, tab, None, flags=flags, scale=1.0)
            got = G.unproject(ctx, depth, tab, None, flags, 1.0)
            assert same_with_nan(got["xyz"], ref_xyz) and np.array_equal(got["valid"], ref_valid)


def test_points_from_xyz16_and_crop(ctx, oracle, nfov2):
    depth, tab, T = nfov2
    _, _, x16 = oracle.unproject(depth[:1, :1], tab[:1], None, flags=1, scale=1.0, want_xyz16=True)
    x16 = x16[0]
    r = np.random.default_rng(1)
    rgb = r.integers(0, 256, (x16.shape[0], 3)).astype(np.uint8)
    rgb[r.random(x16.shape[0]) < 0.6] = 0
    keep_ref, med_ref = oracle.crop_mask(rgb, x16, 750.0)
    keep, med = G.crop_mask(ctx, rgb, x16, 750.0)
    assert med == med_ref and np.array_equal(keep, keep_ref)
    Tm = synth.scale_extrinsics(T, 1.0)[1]
    for Tuse, k in ((None, None), (Tm, keep_ref)):
        ref, rv = oracle.points_from_xyz16(x16, T=Tuse, keep=k)
        got, gv = G.points_from_xyz16(ctx, x16, T=Tuse, keep=k)
        assert same_with_nan(got, ref) and np.array_equal(gv, rv)
    # odd / even medians
    for n in (5, 6, 1, 2):
        a = np.zeros((n, 3), np.int16)
        a[:, 2] = r.integers(-500, 5000, n)
        _, m = G.crop_mask(ctx, np.ones((n, 3), np.uint8), a, 10.0)
        assert m == float(np.median(a[:, 2]))


def test_transform_bounds_compact(ctx, oracle):
    pts = make_surface_cloud(5003, seed=2)
    T = synth.perturbed_extrinsic(synth.extrinsics(3)[1])
    assert np.array_equal(G.transform(ctx, pts, T), oracle.transform(pts, T))
    assert np.array_equal(G.transform(ctx, pts, T, True), oracle.transform(pts, T, True))
    pts[::9] = np.nan
    b, nv = G.bounds(ctx, pts)
    ok = ~np.isnan(pts[:, 0])
    assert nv == ok.sum() and np.array_equal(b, np.concatenate([pts[ok].min(0), pts[ok].max(0)]))
    out, idx, _ = G.compact(ctx, pts)                      # NaN test
    assert np.array_equal(out, pts[ok]) and np.array_equal(idx, np.flatnonzero(ok))
    mask = (np.arange(len(pts)) % 3 == 0).astype(np.uint8)
    col = np.random.default_rng(3).random((len(pts), 3)).astype(np.float32)
    for inv in (False, True):
        sel = mask.astype(bool) != inv
        out, idx, oc = G.compact(ctx, np.nan_to_num(pts), mask, inv, col)
        assert np.array_equal(out, np.nan_to_num(pts)[sel]) and np.array_equal(idx, np.flatnonzero(sel))
        assert np.array_equal(oc, col[sel])
    for m in (np.zeros(len(pts), np.uint8), np.ones(len(pts), np.uint8)):
        out, idx, _ = G.compact(ctx, np.nan_to_num(pts), m)
        assert len(out) == m.sum()



@pytest.mark.parametrize("n", [1, 31, 2047, 2048, 2049, 65536, 300007, 1300003, 6000011])
def test_compact_single_pass_scan_across_tiles(ctx, n):
    """Ordered compaction is one kernel: tiles of 2048 whose offsets come from published tile aggregates and group
    totals (groups of 32 tiles), each word tagged with a per-call epoch (never cleared) -- while the grid is resident at
    once (<= 4 CTAs per SM); larger arrays (the last two sizes) take the count / scan / scatter path.  Ragged sizes around the tile
    and group edges, sparse / dense / run-structured masks, and back-to-back calls on the same context (stale words
    of earlier calls must read as 'not ready')."""
    rng = np.random.default_rng(n)
    pts = rng.random((n, 3), dtype=np.float32)
    masks = [(rng.random(n) < p).astype(np.uint8) for p in (0.001, 0.5, 0.999)]
    masks.append(((np.arange(n) // 777) % 2).astype(np.uint8))      # long runs: whole tiles kept / dropped
    for rep in range(2):
        for m in masks:
            for inv in (False, True):
                sel = m.astype(bool) != inv
                out, idx, _ = G.compact(ctx, pts, m, inv)
                assert np.array_equal(idx, np.flatnonzero(sel)) and np.array_equal(out, pts[sel])

# ------------------------------------------------------------------ K2 ----
@pytest.mark.parametrize("n,voxel,scale", [(50000, 0.05, 1.0), (50000, 35.0, 1000.0), (3000, 0.01, 1.0), (17, 0.5, 1.0)])
def test_voxel_downsample_bit_exact(ctx, oracle, n, voxel, scale):
    pts = make_surface_cloud(n, seed=n, scale=scale)
    r = np.random.default_rng(4)
    col = r.random((n, 3)).astype(np.float32)
    nrm = r.normal(size=(n, 3)).astype(np.float32)
    ref = oracle.voxel_downsample(pts, voxel, col, nrm)
    got = G.voxel(ctx, pts, voxel, col, nrm)
    assert got["m"] == ref["m"]
    assert np.array_equal(got["ijk"], ref["ijk"])                      # voxel keys: bit-exact
    assert np.array_equal(got["point_voxel"], ref["point_voxel"])      # point -> voxel map: bit-exact
    assert np.array_equal(got["min_bound"], ref["min_bound"])
    assert np.array_equal(got["points"], ref["points"])                # means: same op order -> identical
    assert np.array_equal(got["colors"], ref["colors"])
    assert np.allclose(got["normals"], ref["normals"], atol=1e-6)
    assert np.abs(got["points"].astype(np.float64) - ref["points"]).max() <= COORD_TOL * scale
    # canonical order = sorted by (ix, iy, iz)
    key = got["ijk"].astype(np.int64)
    assert np.all(np.lexsort((key[:, 2], key[:, 1], key[:, 0])) == np.arange(len(key)))


def test_voxel_nan_rows_wide_keys_and_errors(ctx, oracle):
    pts = make_surface_cloud(20000, seed=5)
    pts[::6] = np.nan
    ref = oracle.voxel_downsample(pts, 0.03)
    got = G.voxel(ctx, pts, 0.03)
    assert np.array_equal(got["points"], ref["points"]) and np.array_equal(got["point_voxel"], ref["point_voxel"])
    # millimetre data with the reference's 0.02 default (filtering.py:16): 57-bit keys -> 64-bit sort path
    mm = make_surface_cloud(4000, seed=6, scale=3000.0)
    mm[:50] = mm[50:100]                                   # exact duplicates are the only merges
    ref = oracle.voxel_downsample(mm, 0.02)
    got = G.voxel(ctx, mm, 0.02)
    assert got["m"] == ref["m"] and np.array_equal(got["ijk"], ref["ijk"]) and np.array_equal(got["points"], ref["points"])
    from kinectpy_b200 import KinectPyB200Error
    with pytest.raises(KinectPyB200Error):
        G.voxel(ctx, mm, 0.0)
    with pytest.raises(KinectPyB200Error):
        G.voxel(ctx, mm, 1e-7)                             # extent / voxel overflows the key
    assert G.voxel(ctx, np.zeros((0, 3), np.float32), 0.1)["m"] == 0
    allnan = np.full((10, 3), np.nan, np.float32)
    assert G.voxel(ctx, allnan, 0.1)["m"] == 0


# ------------------------------------------------------------------ K3 ----
@pytest.mark.parametrize("n,k,quantum", [(20000, 20, None), (8000, 50, 0.01), (3000, 200, None), (5000, 1, 0.02), (40, 64, None),
                                         (6000, 31, None), (6000, 32, 0.01), (6000, 33, None), (6000, 65, None),
                                         (3000, 1000, None)])
def test_knn_indices_bit_exact(ctx, oracle, n, k, quantum):
    pts = make_surface_cloud(n, seed=100 + k, quantum=quantum, outliers=0.02)
    ri, rd, rc = oracle.knn(pts, k)
    gi, gd, gc = G.knn(ctx, pts, k)
    assert np.array_equal(gc, rc)
    assert np.array_equal(gi, ri)          # canonical (d2, index) order, ties included
    assert np.array_equal(gd, rd)


def test_knn_hybrid_external_queries_and_hints(ctx, oracle):
    pts = make_surface_cloud(15000, seed=7)
    q = make_surface_cloud(3000, seed=8) + np.float32(0.003)
    q[:5] = [[9, 9, 9], [-9, 0, 0], [0, 0, 40], [1.49, 1.49, 1.49], [-1.5, -1.5, -1.5]]   # far outside the grid
    ri, rd, rc = oracle.knn(pts, 30, queries=q, radius=0.07)
    gi, gd, gc = G.knn(ctx, pts, 30, queries=q, radius=0.07)
    assert np.array_equal(gc, rc) and np.array_equal(gi, ri) and np.array_equal(gd, rd)
    ri, rd, rc = oracle.knn(pts, 8, queries=q)
    for hint in (0.0, 0.01, 0.2, 5.0):      # the grid cell changes the cost of the search, never its result
        gi, gd, gc = G.knn(ctx, pts, 8, queries=q, cell_hint=hint)
        assert np.array_equal(gi, ri) and np.array_equal(gd, rd)
    pts[::10] = np.nan                      # absent rows are never returned and get empty results
    ri, rd, rc = oracle.knn(pts, 5)
    gi, gd, gc = G.knn(ctx, pts, 5)
    assert np.array_equal(gc, rc) and np.array_equal(gi, ri)


@pytest.mark.parametrize("n,k,ratio", [(30000, 20, 2.0), (10000, 50, 0.30), (4000, 200, 3.0)])
def test_sor_mask_bit_exact(ctx, oracle, n, k, ratio):
    pts = make_surface_cloud(n, seed=200 + k, outliers=0.01)
    rk, rm, rs = oracle.sor(pts, k, ratio)
    gk, gm, gs, kept = G.sor(ctx, pts, k, ratio)
    assert np.array_equal(gm, rm)           # per-point mean distance: canonical sum -> identical doubles
    assert np.array_equal(gs, rs)           # mu, std, threshold: canonical tree -> identical doubles
    assert np.array_equal(gk, rk) and kept == rk.sum()
    assert 0 < kept < n


def test_sor_edge_cases(ctx, oracle):
    from kinectpy_b200 import KinectPyB200Error
    dup = np.tile(np.array([[1, 2, 3]], np.float32), (40, 1))
    assert G.sor(ctx, dup, 5, 1.0)[3] == 0                 # all means are 0 -> nothing kept
    small = make_surface_cloud(7, seed=9)
    rk, rm, rs = oracle.sor(small, 20, 2.0)                # fewer points than k
    gk, gm, gs, _ = G.sor(ctx, small, 20, 2.0)
    assert np.array_equal(gk, rk) and np.array_equal(gm, rm)
    with pytest.raises(KinectPyB200Error):
        G.sor(ctx, small, 0, 1.0)
    with pytest.raises(KinectPyB200Error):
        G.sor(ctx, small, 5, 0.0)


def test_radius_outlier_bit_exact(ctx, oracle):
    pts = np.array([[0, 0, 0], [1, 0, 0], [2, 0, 0], [10, 0, 0]], np.float32)
    keep, cnt, _ = G.radius_outlier(ctx, pts, 1, 1.0)
    assert cnt.tolist() == [1, 1, 1, 1] and keep.sum() == 0        # strict d2 < r2
    big = make_surface_cloud(20000, seed=10, quantum=0.005)
    for nb, r in ((5, 0.05), (16, 0.03), (1, 0.005)):
        rk, rc = oracle.radius_outlier(big, nb, r)
        gk, gc, kept = G.radius_outlier(ctx, big, nb, r)
        assert np.array_equal(gc, rc) and np.array_equal(gk, rk) and kept == rk.sum()


def test_normals_match_oracle_modulo_sign(ctx, oracle):
    pts = make_surface_cloud(20000, seed=11, outliers=0.005)
    for radius, nn in ((0.06, 30), (0.1, 40), (0.0, 12)):
        ref = oracle.estimate_normals(pts, radius, nn).astype(np.float64)
        got = G.normals(ctx, pts, radius, nn).astype(np.float64)
        assert np.allclose(np.linalg.norm(got, axis=1), 1.0, atol=1e-5)
        dots = np.abs((ref * got).sum(1))
        # near-degenerate neighbourhoods (two close eigenvalues) amplify the last-bit difference of the
        # cumulant sums; everything else agrees to float32 resolution
        assert np.mean(dots > 1 - 1e-6) > 0.999
        assert np.mean(dots > 1 - 1e-3) > 0.9999
    lonely = np.array([[0, 0, 0], [5, 5, 5], [5.001, 5, 5]], np.float32)
    assert G.normals(ctx, lonely, 0.1, 30).tolist() == [[0, 0, 1], [0, 0, 1], [0, 0, 1]]


# ------------------------------------------------------------------ K4 ----
def floor_scene(n, seed, frac_out=0.25):
    r = np.random.default_rng(seed)
    pts = np.stack([r.uniform(-2, 2, n), 1.2 + r.normal(0, 0.003, n), r.uniform(0, 4, n)], 1)
    k = int(n * frac_out)
    pts[:k] = r.uniform(-2, 2, (k, 3))
    return pts.astype(np.float32)


@pytest.mark.parametrize("n,ransac_n,iters", [(40000, 3, 1000), (12000, 30, 2000), (500, 3, 64), (3000, 5, 700)])
def test_ransac_inlier_set_bit_exact(ctx, oracle, n, ransac_n, iters):
    pts = floor_scene(n, seed=n, frac_out=0.25 if ransac_n == 3 else 0.0)
    thr = 0.01
    rp, rmask, rbest, rcounts = oracle.ransac_plane(pts, thr, ransac_n, iters, seed=1234)
    gp, gmask, gbest, gcounts, ninl = G.ransac(ctx, pts, thr, ransac_n, iters, seed=1234)
    assert np.array_equal(gcounts, rcounts)      # every hypothesis' inlier count
    assert gbest == rbest
    assert np.array_equal(gmask, rmask) and ninl == rmask.sum()
    assert np.allclose(gp, rp, rtol=0, atol=1e-9)
    # a different seed gives different hypotheses; same seed is reproducible
    g2 = G.ransac(ctx, pts, thr, ransac_n, iters, seed=99)
    assert not np.array_equal(g2[3], gcounts)
    assert np.array_equal(G.ransac(ctx, pts, thr, ransac_n, iters, seed=1234)[1], gmask)


def test_ransac_degenerate_and_errors(ctx, oracle):
    from kinectpy_b200 import KinectPyB200Error
    line = np.stack([np.arange(100), np.zeros(100), np.zeros(100)], 1).astype(np.float32)   # collinear: no valid plane
    rp, rmask, rbest, _ = oracle.ransac_plane(line, 0.01, 3, 50)
    gp, gmask, gbest, _, ninl = G.ransac(ctx, line, 0.01, 3, 50)
    assert gbest == rbest == -1 and ninl == 0 and gmask.sum() == 0
    with pytest.raises(KinectPyB200Error):
        G.ransac(ctx, line[:2], 0.01, 3, 10)
    with pytest.raises(KinectPyB200Error):
        G.ransac(ctx, line, 0.01, 2, 10)


def test_plane_side_and_band(ctx, oracle):
    pts = make_surface_cloud(30000, seed=12)
    a, b, c, d = 0.3, -0.9, 0.2, 0.05
    m, kept = G.plane_side(ctx, pts, a, b, c, d)
    ref = oracle.plane_side(pts, a, b, c, d)
    assert np.array_equal(m, ref) and kept == ref.sum()
    for axis, band in ((1, 0.2), (2, 0.05), (0, 10.0)):
        lo, amax, nlo = G.band(ctx, pts, band, axis)
        ref = oracle.band_mask(pts, band, axis)
        assert np.array_equal(lo, ref) and nlo == ref.sum() and amax == float(pts[:, axis].max())


# ------------------------------------------------------------------ K5 ----
def icp_case(oracle, n, seed, unit=1.0):
    tgt = make_surface_cloud(n, seed=seed, outliers=0.0, scale=unit)
    nrm = oracle.estimate_normals(tgt, 0.08 * unit, 30)
    D = synth.perturbed_extrinsic(np.eye(4), angle_deg=1.0, shift_mm=(5, -5, 5), unit_scale=1e-3 * unit)
    src = oracle.transform(tgt[::2] + 0, np.linalg.inv(D))
    return src, tgt, nrm, D


@pytest.mark.parametrize("n,max_iter,unit", [(20000, 30, 1.0), (6000, 5, 1.0), (20000, 30, 1000.0), (6000, 0, 1.0)])
def test_icp_matches_oracle(ctx, oracle, n, max_iter, unit):
    src, tgt, nrm, D = icp_case(oracle, n, seed=300 + n, unit=unit)
    ref = oracle.icp_point_to_plane(src, tgt, nrm, 0.05 * unit, init=np.eye(4), max_iter=max_iter)
    got = G.icp(ctx, src, tgt, nrm, 0.05 * unit, init=np.eye(4), max_iter=max_iter)
    assert got["iters"] == ref["iters"]
    assert got["ncorr"] == ref["ncorr"]
    assert np.abs(got["T"][:3, :3] - ref["T"][:3, :3]).max() < ICP_TOL
    assert np.abs(got["T"][:3, 3] - ref["T"][:3, 3]).max() < ICP_TOL * unit
    assert got["fitness"] == pytest.approx(ref["fitness"], abs=1e-9)
    assert got["rmse"] == pytest.approx(ref["rmse"], rel=1e-6, abs=1e-9 * unit)
    if max_iter >= 30:                       # and both recover the planted transform
        assert np.abs(got["T"][:3, :3] - D[:3, :3]).max() < 2e-3
        assert np.abs(got["T"][:3, 3] - D[:3, 3]).max() < 2e-3 * unit


def test_icp_no_overlap_and_errors(ctx, oracle):
    from kinectpy_b200 import KinectPyB200Error
    src, tgt, nrm, _ = icp_case(oracle, 3000, seed=13)
    far = src + np.float32(50.0)
    ref = oracle.icp_point_to_plane(far, tgt, nrm, 0.05, max_iter=30)
    got = G.icp(ctx, far, tgt, nrm, 0.05, max_iter=30)
    assert got["ncorr"] == ref["ncorr"] == 0 and got["fitness"] == 0 and np.array_equal(got["T"], np.eye(4))
    assert got["iters"] == ref["iters"]
    with pytest.raises(KinectPyB200Error):
        G.icp(ctx, src, tgt, nrm, 0.0)


# ------------------------------------------------- run-to-run determinism --
def test_outputs_are_deterministic(ctx):
    pts = make_surface_cloud(60000, seed=14, outliers=0.02)
    a = (G.voxel(ctx, pts, 0.02), G.sor(ctx, pts, 20, 2.0), G.knn(ctx, pts, 16), G.normals(ctx, pts, 0.05, 30))
    b = (G.voxel(ctx, pts, 0.02), G.sor(ctx, pts, 20, 2.0), G.knn(ctx, pts, 16), G.normals(ctx, pts, 0.05, 30))
    assert np.array_equal(a[0]["points"], b[0]["points"]) and np.array_equal(a[0]["ijk"], b[0]["ijk"])
    assert np.array_equal(a[1][0], b[1][0]) and np.array_equal(a[1][1], b[1][1])
    assert np.array_equal(a[2][0], b[2][0]) and np.array_equal(a[2][1], b[2][1])
    assert np.array_equal(a[3], b[3])
