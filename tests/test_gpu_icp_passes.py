"""The per-call ICP kernels (``kp_icp_point_to_plane``, ``kp_icp_point_to_point``, ``kp_icp_colored``) held pass by
pass to the float64 reference of ``tests/icp_ref64.py`` (itself pinned to the oracle by ``test_oracle_icp_passes.py``).

The state after pass k is the entry point's result for ``max_iter = k`` and ``rel_fit = rel_rmse = -1``; it is compared
for k = 0, 1, 2, 5 and for the converged run with the default thresholds:

* ncorr, fitness and iters equal;
* rmse within RMSE_TOL relative (the sums of d² differ only in order);
* T within T_TOL, the translation divided by the unit of the case (metres 1, millimetres 1000).

Where the system is singular by construction (one or two matches) the reference's LU and the kernel's scalar
elimination return different rounding residues, so the kernel is held to the oracle there, bit for bit: with two terms
every sum is the same in any order, and the elimination performs the oracle's operations.

Largest gaps observed on a B200 (1000 W), over every case of this file: rmse 1.62e-15 relative, T 3.64e-14.  The bars
are kept within 100x of that: RMSE_TOL = 1e-13 (summation order alone, about sqrt(n) eps for 1e6 terms) and
T_TOL = 3e-12.  Each run prints the largest gaps it saw."""
import numpy as np
import pytest

import icp_cases as IC
import icp_ref64 as R

pytestmark = pytest.mark.gpu

RMSE_TOL = 1e-13
T_TOL = 3e-12
KS = (0, 1, 2, 5)
GAPS = {"rmse_rel": 0.0, "T": 0.0}


@pytest.fixture(scope="module", autouse=True)
def report_gaps():
    yield
    print("\n[icp passes] largest gaps: rmse %.3g relative (bar %.0e), T %.3g (bar %.0e)"
          % (GAPS["rmse_rel"], RMSE_TOL, GAPS["T"], T_TOL))


def gpu(ctx, c, mode, k, lam=0.968, rel=-1.0):
    import gpu_helpers as G
    a = dict(init=c["init"], max_iter=k, rel_fit=rel, rel_rmse=rel)
    if mode == R.PLANE:
        return G.icp(ctx, c["src"], c["tgt"], c["tgt_n"], c["max_corr"], **a)
    if mode == R.POINT:
        return G.icp_p2p(ctx, c["src"], c["tgt"], c["max_corr"], **a)
    return G.icp_colored(ctx, c["src"], c["src_col"], c["tgt"], c["tgt_col"], c["tgt_n"], c["max_corr"], lam=lam, **a)


def oracle_run(orc, c, mode, k, lam=0.968, rel=-1.0):
    a = dict(init=c["init"], max_iter=k, rel_fit=rel, rel_rmse=rel)
    if mode == R.PLANE:
        return orc.icp_point_to_plane(c["src"], c["tgt"], c["tgt_n"], c["max_corr"], **a)
    if mode == R.POINT:
        return orc.icp_point_to_point(c["src"], c["tgt"], c["max_corr"], **a)
    return orc.icp_colored(c["src"], c["src_col"], c["tgt"], c["tgt_col"], c["tgt_n"], c["max_corr"], lambda_geometric=lam, **a)


class Ref:
    """The reference's passes of one case, produced on demand."""

    def __init__(self, ctx, c, mode, lam=0.968):
        kw = {}
        if mode == R.COLORED:
            import gpu_helpers as G
            # the gradient the kernel computes internally (kp_color_gradient on the same inputs), so the pass is
            # tested in isolation
            kw = dict(src_colors=c["src_col"], tgt_colors=c["tgt_col"], lam=lam,
                      tgt_grad=G.color_gradient(ctx, c["tgt"], c["tgt_col"], c["tgt_n"], 2.0 * c["max_corr"], 30))
        self.gen = R.passes(c["src"], c["tgt"], c["max_corr"], init=c["init"], mode=mode, tgt_normals=c.get("tgt_n"), **kw)
        self.recs = []

    def __getitem__(self, k):
        while len(self.recs) <= k:
            self.recs.append(next(self.gen))
        return self.recs[k]

    def converged(self, max_iter=30, rel=1e-6):
        k = 0
        while k < max_iter and not (k > 0 and abs(self[k - 1]["fitness"] - self[k]["fitness"]) < rel
                                    and abs(self[k - 1]["rmse"] - self[k]["rmse"]) < rel):
            k += 1
        return self[k]


def same(got, rec, c, iters, T_tol=T_TOL):
    assert got["ncorr"] == rec["ncorr"] and got["fitness"] == rec["fitness"] and got["iters"] == iters, \
        (got["ncorr"], rec["ncorr"], got["iters"], iters)
    g = abs(got["rmse"] - rec["rmse"]) / rec["rmse"] if rec["rmse"] else abs(got["rmse"])
    GAPS["rmse_rel"] = max(GAPS["rmse_rel"], g)
    assert g <= RMSE_TOL, g
    d = np.abs(got["T"] - rec["T"])
    d[:3, 3] /= c["unit"]
    if T_tol is not None:
        GAPS["T"] = max(GAPS["T"], d.max())
        assert d.max() <= T_tol, d.max()


def run_case(ctx, c, mode=R.PLANE, ks=KS, lam=0.968, converged=True):
    ref = Ref(ctx, c, mode, lam)
    for k in ks:
        same(gpu(ctx, c, mode, k, lam), ref[k], c, k)
    if converged:
        rec = ref.converged()
        same(gpu(ctx, c, mode, 30, lam, rel=1e-6), rec, c, rec["pass"])
    return ref


# ---------------------------------------------------------------------------------------- 1. hand-over shapes
# 256 points per CTA, 32 CTAs per group: 1, 2, 32 and 33 CTAs; exactly 32 groups; 33 groups (the final fold takes more
# than 32 rows); 129 groups
@pytest.mark.parametrize("n", [1, 255, 256, 257, 8191, 8192, 8193, 262144, 262145, 1050000])
def test_handover_shapes_point_to_plane(ctx, n):
    run_case(ctx, IC.surface_pair(n, seed=n))


@pytest.mark.parametrize("mode", [R.POINT, R.COLORED], ids=["point", "colored"])
@pytest.mark.parametrize("n", [257, 8193, 262145])
def test_handover_shapes_other_modes(ctx, mode, n):
    run_case(ctx, IC.surface_pair(n, seed=n), mode)


# ---------------------------------------------------------------------------------------- 2. the gate
def test_gate_faces_edges_corners_and_far_points(ctx):
    """d² == r² exactly is out, one ulp inside is in, beyond every face, edge and corner of the target's box (cells at
    -1 and past the end), plus points 1e3 and 1e6 away."""
    c = IC.gate_case()
    ref = run_case(ctx, c)
    assert ref[0]["ncorr"] == 2 * 26


def test_target_of_one_point(ctx, oracle):
    c = IC.one_point_target()
    ref = Ref(ctx, c, R.PLANE)
    same(gpu(ctx, c, R.PLANE, 0), ref[0], c, 0)
    assert ref[0]["ncorr"] == 2
    for k in (1, 2, 5):                        # two matches: a singular system, held to the oracle bit for bit
        got, o = gpu(ctx, c, R.PLANE, k), oracle_run(oracle, c, R.PLANE, k)
        assert got["ncorr"] == o["ncorr"] and got["rmse"] == o["rmse"] and np.array_equal(got["T"], o["T"]), k


# ---------------------------------------------------------------------------------------- 3. ties
def test_ties_go_to_the_lower_index(ctx):
    c = IC.ties_case()
    run_case(ctx, c)


# ---------------------------------------------------------------------------------------- 4. NaN rows, nothing to match
def test_nan_rows(ctx):
    run_case(ctx, IC.nan_case(30000, seed=3))


@pytest.mark.parametrize("which", ["all_nan", "empty_src", "empty_tgt"])
@pytest.mark.parametrize("mode", [R.PLANE, R.POINT, R.COLORED], ids=["plane", "point", "colored"])
def test_nothing_to_match(ctx, mode, which):
    c = IC.surface_pair(300, seed=4)
    c["init"] = IC.rot(0.1, -0.2, 0.3)
    c["init"][:3, 3] = (0.01, 0.02, -0.03)
    if which == "all_nan":
        c["src"][:] = np.nan
    elif which == "empty_src":
        c["src"], c["src_col"] = c["src"][:0], c["src_col"][:0]
    else:
        c["tgt"], c["tgt_n"], c["tgt_col"] = c["tgt"][:0], c["tgt_n"][:0], c["tgt_col"][:0]
    for k in (0, 1, 5):
        got = gpu(ctx, c, mode, k)
        assert got["ncorr"] == 0 and got["fitness"] == 0.0 and got["rmse"] == 0.0 and np.array_equal(got["T"], c["init"])


# ---------------------------------------------------------------------------------------- 5. far from the origin
@pytest.mark.parametrize("unit", [1.0, 1000.0], ids=["m", "mm"])
def test_far_from_the_origin(ctx, unit):
    """The surface 1e4 units from the origin, where the fp32 spacing (1e-3 units) is ~3 % of max_corr, under an init
    that is not dyadic (a small rotation about the cloud plus a translation): the moving source is then a double that
    its fp32 copy misses by up to half an ulp, so the pre-test's fp32 distances are off by a sizeable fraction of d²
    and only the slack keeps every candidate that can win.  A lost candidate changes a partner and with it the rmse.
    (Pass 0 only, where T is still the init: 1e4 units from the centre of rotation the 6x6 system is too
    ill-conditioned for a pass-by-pass comparison after an update to mean anything.)"""
    c = IC.surface_pair(30000, seed=17, unit=unit, offset=1e4 * unit)
    c["init"] = IC.about(IC.rot(1e-4, -2e-4, 1.5e-4), np.full(3, 1e4 * unit), np.array([3e-3, -2e-3, 1e-3]) * unit)
    ref = Ref(ctx, c, R.PLANE)
    same(gpu(ctx, c, R.PLANE, 0), ref[0], c, 0)
    assert ref[0]["ncorr"] > 0.99 * len(c["src"])
    cur = R.affine(c["init"], c["src"].astype(np.float64))
    assert np.abs(cur - cur.astype(np.float32)).max() > 0.005 * c["max_corr"]     # the fp32 copy is far off


# ---------------------------------------------------------------------------------------- 6. degenerate systems
def test_planar_zero_residual_keeps_init(ctx):
    c = IC.planar_case()
    ref = run_case(ctx, c)
    for k in KS:
        got = gpu(ctx, c, R.PLANE, k)
        assert got["ncorr"] == 300 and np.array_equal(got["T"], np.eye(4)) and not ref[k]["b"].any(), k


def test_no_match_is_the_identity_update(ctx):
    c = IC.surface_pair(2000, seed=6)
    c["src"] = c["src"] + np.float32(50.0)
    for k in KS:
        got = gpu(ctx, c, R.PLANE, k)
        assert got["ncorr"] == 0 and np.array_equal(got["T"], np.eye(4))


@pytest.mark.parametrize("mode", [R.PLANE, R.POINT, R.COLORED], ids=["plane", "point", "colored"])
@pytest.mark.parametrize("nmatch", [1, 2])
def test_one_and_two_matches_equal_the_oracle(ctx, oracle, mode, nmatch):
    """Sums of one or two terms are the same in any order, so the kernel's T equals the oracle's bit for bit (coloured
    with two matches at lambda = 0: with both rows present the oracle adds the photometric products before the
    geometric ones of the same point, the kernel per point, so the two-term sums group differently).  Point-to-point
    with two matches is rank 1 and compared on the moved matched rows."""
    c = IC.few_matches_case(nmatch)
    lam = 0.0 if (mode == R.COLORED and nmatch == 2) else 0.968
    s = c["src"][:nmatch].astype(np.float64)            # the matched rows (the others are far away)
    for k in KS:
        got, o = gpu(ctx, c, mode, k, lam), oracle_run(oracle, c, mode, k, lam)
        assert got["ncorr"] == o["ncorr"] and got["fitness"] == o["fitness"] and got["iters"] == o["iters"], k
        if mode == R.POINT and nmatch == 2:
            assert np.abs(R.affine(got["T"], s) - R.affine(o["T"], s)).max() < 1e-9, k
        else:
            assert got["rmse"] == o["rmse"] and np.array_equal(got["T"], o["T"]), k


@pytest.mark.parametrize("axis_aligned", [True, False], ids=["axis", "general"])
def test_collinear_point_to_point(ctx, axis_aligned):
    """Rank-1 cross-covariance: the rotation about the line is free, so the moved source is compared (along the x axis
    the cross-covariance has exact zeros, and only the rank-1 completion of kp_umeyama gives a finite rotation)."""
    c = IC.collinear_case(axis_aligned)
    ref = Ref(ctx, c, R.POINT)
    s = c["src"].astype(np.float64)
    for k in KS:
        got = gpu(ctx, c, R.POINT, k)
        assert got["ncorr"] == ref[k]["ncorr"] and got["iters"] == k
        assert np.isfinite(got["T"]).all() and abs(np.linalg.det(got["T"][:3, :3]) - 1) < 1e-12
        assert np.abs(R.affine(got["T"], s) - R.affine(ref[k]["T"], s)).max() < 1e-6, k


def test_coplanar_point_to_point_is_a_rotation(ctx):
    c = IC.coplanar_reflection_case()
    ref = run_case(ctx, c, R.POINT)
    assert abs(np.linalg.det(ref[5]["T"][:3, :3]) - 1) < 1e-12


# ---------------------------------------------------------------------------------------- 7. coloured lambda
@pytest.mark.parametrize("lam", [0.0, 0.5, 0.968, 1.0])
def test_colored_lambda(ctx, lam):
    """Coloured ICP on the bumpy textured surface, whose JᵀJ stays well conditioned at every lambda (condition number
    at pass 0: 289 at lambda 0, 3.01 at 0.5, 51 at 0.968, 551 at 1)."""
    c = IC.surface_pair(20000, seed=29)
    ref = run_case(ctx, c, R.COLORED, lam=lam)
    cond = np.linalg.cond(ref[0]["A"])
    print("\n[icp passes] coloured lambda %.3f: cond(JtJ) at pass 0 = %.3g" % (lam, cond))
    assert cond < 1e3                                   # measured: 289, 3.01, 51, 551 for the four lambdas


# ---------------------------------------------------------------------------------------- 8. pass batching across calls
def test_pass_batching_across_calls(ctx):
    """kp_icp_device sizes its first batch of launches from the previous call on the context (passes + 2), then adds
    batches of 6, and stops fetching once the device state says `done`.  A sequence of calls on one context must give
    what each call gives on a fresh context.  p is the pass the default thresholds converge at (from the reference):
    the converged calls are preceded by calls that set the hint so that convergence falls on the last launch of the
    first batch, and on the first launch of the second."""
    from kinectpy_b200 import _cabi
    c = IC.surface_pair(20000, seed=31)
    c["init"] = IC.rot(0.05, -0.05, 0.05)
    c["init"][:3, 3] = (0.03, -0.03, 0.03)
    p = Ref(ctx, c, R.PLANE).converged()["pass"]
    assert p >= 3
    seq = [(2, -1.0),        # 3 passes (fresh context: first batch 16, clipped to 3)
           (20, -1.0),       # 21 passes: first batch 5, then 6, 6, 6 (four fetch rounds)
           (22, -1.0),       # 23 passes: exactly the first batch (21 + 2)
           (30, -1.0),       # 31 passes: first batch 25, then one of 6 ending exactly at the last pass
           (p - 2, -1.0),    # p - 1 passes: the next first batch is p + 1 launches ...
           (30, 1e-6),       # ... and this call converges at pass p, the batch's last launch (done, not max_iter)
           (p - 3, -1.0),    # p - 2 passes: the next first batch is p launches ...
           (30, 1e-6),       # ... and this call converges at pass p, the first launch of the second batch
           (0, -1.0)]
    shared = _cabi.Context()
    try:
        for k, rel in seq:
            a = gpu(shared, c, R.PLANE, k, rel=rel)
            fresh = _cabi.Context()
            try:
                b = gpu(fresh, c, R.PLANE, k, rel=rel)
            finally:
                fresh.close()
            assert a["iters"] == b["iters"] and a["ncorr"] == b["ncorr"], (k, rel)
            assert a["fitness"] == b["fitness"] and a["rmse"] == b["rmse"] and np.array_equal(a["T"], b["T"]), (k, rel)
            assert a["iters"] == (k if rel < 0 else p), (k, rel)
    finally:
        shared.close()
