"""Global registration (SURVEY.md 8f, row f3): compute_fpfh_feature and
registration_ransac_based_on_feature_matching behind execute_global_registration
(preprocessing/registration.py:15-21, 32-62).  CPU tests pin the oracle against brute-force numpy; GPU tests
compare the kernels with the oracle: matches and RANSAC bookkeeping exactly, features and transforms within
tolerance (CUDA's and glibc's acos / atan2 differ in the last bit, which can move a sample across a bin edge)."""
import numpy as np
import pytest

from kinectpy_b200 import synth


def bumpy_scene(n, seed):
    """A surface with enough distinctive relief for features to be discriminative, plus a box corner."""
    r = np.random.default_rng(seed)
    u = r.uniform(-1, 1, (n, 2))
    z = (0.25 * np.exp(-((u[:, 0] - 0.3) ** 2 + (u[:, 1] + 0.2) ** 2) / 0.05) - 0.2 * np.exp(-((u[:, 0] + 0.5) ** 2 + (u[:, 1] - 0.4) ** 2) / 0.03)
         + 0.1 * np.sin(4 * u[:, 0]) * np.cos(3 * u[:, 1]) + 0.15 * (u[:, 0] > 0.55) + 0.1 * (u[:, 1] < -0.6))
    pts = np.stack([u[:, 0], u[:, 1], z], axis=1) + r.normal(0, 0.0015, (n, 3))
    return pts.astype(np.float32)


def pair_features_numpy(p1, n1, p2, n2):
    d = p2 - p1
    L = np.linalg.norm(d)
    if L == 0:
        return np.zeros(3)
    a1, a2 = n1 @ d / L, n2 @ d / L
    if np.arccos(abs(a1)) > np.arccos(abs(a2)):
        n1, n2, d, f2 = n2, n1, -d, -a2
    else:
        f2 = a1
    v = np.cross(d, n1)
    vn = np.linalg.norm(v)
    if vn == 0:
        return np.zeros(3)
    v = v / vn
    w = np.cross(n1, v)
    return np.array([np.arctan2(w @ n2, n1 @ n2), v @ n2, f2])


def fpfh_numpy(pts, nrm, radius, max_nn, rows):
    """Brute-force restatement of Open3D's SPFH / FPFH for a few rows."""
    P, N = pts.astype(np.float64), nrm.astype(np.float64)

    def nbrs(i):
        d2 = ((P - P[i]) ** 2).sum(1)
        d2 = (P[:, 0] - P[i, 0]) ** 2 + (P[:, 1] - P[i, 1]) ** 2
        d2 = d2 + (P[:, 2] - P[i, 2]) ** 2
        order = np.lexsort((np.arange(len(P)), d2))
        order = order[d2[order] < radius * radius][:max_nn]
        return order, d2[order]

    def spfh(i):
        h = np.zeros(33)
        idx, _ = nbrs(i)
        if len(idx) > 1:
            inc = 100.0 / (len(idx) - 1)
            for j in idx[1:]:
                f = pair_features_numpy(P[i], N[i], P[j], N[j])
                h[int(np.clip(np.floor(11 * (f[0] + np.pi) / (2 * np.pi)), 0, 10))] += inc
                h[11 + int(np.clip(np.floor(11 * (f[1] + 1.0) * 0.5), 0, 10))] += inc
                h[22 + int(np.clip(np.floor(11 * (f[2] + 1.0) * 0.5), 0, 10))] += inc
        return h

    out = []
    for i in rows:
        idx, d2 = nbrs(i)
        f = np.zeros(33)
        if len(idx) > 1:
            s = np.zeros(3)
            for j, dd in zip(idx[1:], d2[1:]):
                if dd == 0:
                    continue
                val = spfh(j) / dd
                f += val
                s += val.reshape(3, 11).sum(1)
            s = np.where(s != 0, 100.0 / np.where(s != 0, s, 1), 0)
            f = f * np.repeat(s, 11) + spfh(i)
        out.append(f)
    return np.array(out)


# ------------------------------------------------------------------ oracle (CPU)
def test_oracle_fpfh_vs_numpy_bruteforce(oracle):
    pts = bumpy_scene(3000, 1)
    nrm = oracle.estimate_normals(pts, 0.08, 30)
    feat = oracle.fpfh(pts, nrm, 0.15, 40)
    assert feat.shape == (3000, 33)
    rows = [0, 17, 555, 1234, 2999]
    ref = fpfh_numpy(pts, nrm, 0.15, 40, rows)
    assert np.abs(feat[rows] - ref).max() < 1e-6 * max(1.0, np.abs(ref).max())
    # each of the three sub-histograms of an interior point sums to ~200 (100 weighted blend + 100 own SPFH)
    sums = feat.reshape(3000, 3, 11).sum(2)
    assert np.allclose(sums[rows], 200.0, atol=1e-6)
    # an isolated point has an all-zero feature
    lonely = np.vstack([pts, np.float32([[50, 50, 50]])])
    nl = np.vstack([nrm, np.float32([[0, 0, 1]])])
    assert not oracle.fpfh(lonely, nl, 0.15, 40)[-1].any()


def test_oracle_feature_match_and_mutual_filter(oracle):
    r = np.random.default_rng(2)
    fb = r.random((500, 33))
    fa = fb[r.permutation(500)[:300]] + r.normal(0, 1e-3, (300, 33))
    fa[10] = fb[3]; fb[7] = fb[3]                      # an exact tie: the lower index wins
    nn, d2 = oracle.feature_match(fa, fb)
    bf = ((fa[:, None, :] - fb[None, :, :]) ** 2).sum(2)
    assert np.array_equal(nn, bf.argmin(1)) and nn[10] == 3
    assert np.allclose(d2, bf.min(1), rtol=1e-12, atol=1e-15)
    nn_ts, _ = oracle.feature_match(fb, fa)
    cor = oracle.mutual_correspondences(nn, nn_ts, True, 3)
    assert len(cor) > 250 and all(nn_ts[j] == i for i, j in cor)
    assert len(oracle.mutual_correspondences(nn, nn_ts, False, 3)) == 300
    # too few mutual pairs: fall back to the unfiltered set
    assert len(oracle.mutual_correspondences(nn[:5], nn_ts, True, 3)) == 5


def test_oracle_ransac_correspondence_recovers_planted_transform(oracle):
    r = np.random.default_rng(3)
    tgt = bumpy_scene(2000, 4)
    D = synth.perturbed_extrinsic(np.eye(4), angle_deg=35.0, shift_mm=(400, -250, 150), unit_scale=1e-3)
    src = oracle.transform(tgt, np.linalg.inv(D))
    cor = np.stack([np.arange(2000), np.arange(2000)], axis=1).astype(np.int32)
    bad = r.random(2000) < 0.6                          # 60 % wrong matches
    cor[bad, 1] = r.integers(0, 2000, bad.sum())
    res = oracle.ransac_correspondence(src, tgt, cor, 0.02, max_iter=20000, seed=5)
    assert res["fitness"] > 0.35 and np.abs(res["T"] - D).max() < 2e-2
    assert 0 <= res["best_iter"] < 20000 and 0 < res["validated"] < 20000
    # early exit: with a high inlier ratio the winner is found within the first few hundred hypotheses
    clean = oracle.ransac_correspondence(src, tgt, cor[~bad], 0.02, max_iter=20000, seed=5)
    assert clean["fitness"] > 0.99 and clean["best_iter"] < 50
    # the checkers reject everything when the clouds are unrelated in scale
    none = oracle.ransac_correspondence(src * 3.0, tgt, cor[~bad], 0.02, max_iter=2000, seed=5)
    assert none["fitness"] == 0.0 and none["validated"] == 0 and np.array_equal(none["T"], np.eye(4))


def test_reference_surface_exposes_global_registration():
    from kinectpy_b200 import o3d
    reg = o3d.pipelines.registration
    for name in ("compute_fpfh_feature", "registration_ransac_based_on_feature_matching", "CorrespondenceCheckerBasedOnEdgeLength",
                 "CorrespondenceCheckerBasedOnDistance", "RANSACConvergenceCriteria", "Feature"):
        assert hasattr(reg, name)
    c = reg.RANSACConvergenceCriteria(250000, 0.999)
    assert (c.max_iteration, c.confidence) == (250000, 0.999)


# ------------------------------------------------------------------ GPU parity
@pytest.mark.gpu
@pytest.mark.parametrize("max_nn", [40, 100])
def test_gpu_fpfh_matches_oracle(ctx, oracle, max_nn):
    import gpu_helpers as G
    pts = bumpy_scene(12000, 6)
    pts[::301] = np.nan
    nrm = oracle.estimate_normals(pts, 0.06, 30)
    ref = oracle.fpfh(pts, nrm, 0.12, max_nn)
    got = G.fpfh(ctx, pts, nrm, 0.12, max_nn)
    # identical up to samples that sit on a bin edge of acos / atan2 (last-bit differences between CUDA and glibc)
    close = np.abs(got - ref).max(axis=1) < 1e-9 * max(1.0, np.abs(ref).max())
    assert close.mean() > 0.995
    assert np.abs(got - ref).max() < 15.0               # a moved sample changes a bin by at most 100 / (nn - 1) twice


@pytest.mark.gpu
def test_gpu_feature_match_bit_exact(ctx, oracle):
    import gpu_helpers as G
    r = np.random.default_rng(8)
    fb = r.random((7001, 33)) * 100
    fa = np.vstack([fb[r.permutation(7001)[:3000]] + r.normal(0, 0.05, (3000, 33)), r.random((333, 33)) * 100])
    fa[5] = fb[11]; fb[4000] = fb[11]
    ref_nn, ref_d2 = oracle.feature_match(fa, fb)
    got_nn, got_d2 = G.feature_match(ctx, fa, fb)
    assert np.array_equal(got_nn, ref_nn) and np.array_equal(got_d2, ref_d2) and got_nn[5] == 11


@pytest.mark.gpu
def test_gpu_ransac_correspondence_matches_oracle(ctx, oracle):
    import gpu_helpers as G
    r = np.random.default_rng(9)
    tgt = bumpy_scene(5000, 10)
    D = synth.perturbed_extrinsic(np.eye(4), angle_deg=50.0, shift_mm=(300, 200, -100), unit_scale=1e-3)
    src = oracle.transform(tgt, np.linalg.inv(D))
    cor = np.stack([np.arange(5000), np.arange(5000)], axis=1).astype(np.int32)
    bad = r.random(5000) < 0.7
    cor[bad, 1] = r.integers(0, 5000, bad.sum())
    for seed, iters in ((1, 50000), (2, 250000)):
        ref = oracle.ransac_correspondence(src, tgt, cor, 0.02, max_iter=iters, seed=seed)
        got = G.ransac_correspondence(ctx, src, tgt, cor, 0.02, max_iter=iters, seed=seed)
        assert got["validated"] == ref["validated"] and got["best_iter"] == ref["best_iter"]
        assert abs(got["fitness"] - ref["fitness"]) <= 1.0 / len(cor) and np.abs(got["T"] - ref["T"]).max() < 1e-9
        assert np.abs(got["T"] - D).max() < 2e-2
    # kp_umeyama on more than three rows, each checker off (edge_sim <= 0, dist_thr <= 0), and the early exit at its
    # ends: confidence 0 stops after the first valid hypothesis, confidence 1 never stops early
    for ransac_n, edge_sim, dist_thr, conf, iters in ((4, 0.95, None, 0.999, 50000), (8, 0.95, None, 0.999, 50000),
                                                      (3, 0.0, None, 0.999, 20000), (4, -1.0, None, 0.999, 20000),
                                                      (3, 0.95, 0.0, 0.999, 20000), (8, 0.95, -1.0, 0.999, 20000),
                                                      (3, 0.95, None, 0.0, 20000), (4, 0.95, None, 1.0, 20000)):
        a = dict(ransac_n=ransac_n, edge_sim=edge_sim, dist_thr=dist_thr, confidence=conf, max_iter=iters, seed=3)
        ref = oracle.ransac_correspondence(src, tgt, cor, 0.02, **a)
        got = G.ransac_correspondence(ctx, src, tgt, cor, 0.02, **a)
        assert got["validated"] == ref["validated"] and got["best_iter"] == ref["best_iter"], a
        assert abs(got["fitness"] - ref["fitness"]) <= 1.0 / len(cor) and np.abs(got["T"] - ref["T"]).max() < 1e-9, a
        assert ref["validated"] > 0
    # degenerate inputs
    z = G.ransac_correspondence(ctx, src, tgt, cor[:2], 0.02, max_iter=100)
    assert z["fitness"] == 0 and np.array_equal(z["T"], np.eye(4))
    from kinectpy_b200 import KinectPyB200Error
    with pytest.raises(KinectPyB200Error):
        G.ransac_correspondence(ctx, src, tgt, cor, 0.02, ransac_n=2)


@pytest.mark.gpu
def test_gpu_execute_global_registration_end_to_end(oracle):
    """The reference call: two views of one scene, no initial guess -> the sub -> master transform (millimetres)."""
    from kinectpy_b200 import o3d
    from kinectpy_b200.preprocessing import registration as R
    scene = bumpy_scene(60000, 12).astype(np.float64) * 1000.0
    D = synth.perturbed_extrinsic(np.eye(4), angle_deg=25.0, shift_mm=(300, -200, 100), unit_scale=1.0)
    r = np.random.default_rng(13)
    master = o3d.geometry.PointCloud(); master.points = scene[r.random(len(scene)) < 0.7]
    sub_pts = scene[r.random(len(scene)) < 0.7]
    sub = o3d.geometry.PointCloud(); sub.points = (sub_pts - D[:3, 3]) @ D[:3, :3]
    o3d.utility.random.seed(7)
    down, feat = R.preprocess_point_cloud(master, 35, 30, 100)
    assert feat.data.shape == (33, len(down)) and feat.dimension() == 33 and feat.num() == len(down)
    T = R.execute_global_registration(master, sub, voxel_size=35, ransac_n_trials=3)
    assert T is not None and np.abs(T[:3, :3] - D[:3, :3]).max() < 0.05 and np.abs(T[:3, 3] - D[:3, 3]).max() < 35.0
    # ...and the refinement the reference runs next brings it home
    T2 = R.execute_point_to_plane_registration(master, sub, T, voxel_size=35)
    assert np.abs(T2[:3, :3] - D[:3, :3]).max() < 5e-3 and np.abs(T2[:3, 3] - D[:3, 3]).max() < 5.0
