"""The float64 pass-by-pass ICP reference (``tests/icp_ref64.py``) pinned to the oracle's ICP loop on the CPU.

The oracle run with ``max_iter = k`` and ``rel_fit = rel_rmse = -1`` stops after pass k; the reference's pass k must
have the same ncorr and fitness, rmse within 1e-12 relative and T within 1e-9.  The oracle so vouches for the
reference's rules on the cases that decide them: NaN rows (absent, but counted in n_src), the strict gate d² < r²
(pairs at d² == r² exactly and one ulp inside), ties to the lower target index (duplicated targets with per-index
normals, sources equidistant to eight lattice points), the zero-residual planar system (T stays init exactly).

With one match, point-to-plane has a rank-1 system that both solvers reject and point-to-point a zero
cross-covariance, so T stays init bit for bit.  With two matches (and with one coloured match) the 6×6 system has
rank ≤ 4 and its solution is the rounding residue of whichever elimination solves it, so only pass 0 is compared
there (``test_gpu_icp_passes.py`` holds the device to the oracle's elimination bit for bit).  Collinear point-to-point matches leave the rotation about the line free: compared on the moved source."""
import numpy as np
import pytest

import icp_cases as IC
import icp_ref64 as R

KS = (0, 1, 2, 5)


def oracle_run(orc, c, mode, k, lam=0.968):
    a = dict(init=c["init"], max_iter=k, rel_fit=-1.0, rel_rmse=-1.0)
    if mode == R.PLANE:
        return orc.icp_point_to_plane(c["src"], c["tgt"], c["tgt_n"], c["max_corr"], **a)
    if mode == R.POINT:
        return orc.icp_point_to_point(c["src"], c["tgt"], c["max_corr"], **a)
    return orc.icp_colored(c["src"], c["src_col"], c["tgt"], c["tgt_col"], c["tgt_n"], c["max_corr"], lambda_geometric=lam, **a)


def ref_passes(orc, c, mode, n, lam=0.968):
    kw = {}
    if mode == R.COLORED:
        _, grad = orc.color_gradient(c["tgt"], c["tgt_col"], c["tgt_n"], 2.0 * c["max_corr"], 30)
        kw = dict(src_colors=c["src_col"], tgt_colors=c["tgt_col"], tgt_grad=grad, lam=lam)
    g = R.passes(c["src"], c["tgt"], c["max_corr"], init=c["init"], mode=mode, tgt_normals=c.get("tgt_n"), **kw)
    return [next(g) for _ in range(n)]


def check(orc, c, mode=R.PLANE, ks=KS, lam=0.968, T_tol=1e-9, exact_T=False, rmse_abs=0.0):
    recs = ref_passes(orc, c, mode, max(ks) + 1, lam)
    for k in ks:
        o, r = oracle_run(orc, c, mode, k, lam), recs[k]
        assert o["ncorr"] == r["ncorr"] and o["fitness"] == r["fitness"] and o["iters"] == k, k
        assert abs(o["rmse"] - r["rmse"]) <= 1e-12 * r["rmse"] + rmse_abs, k
        if exact_T:
            assert np.array_equal(o["T"], r["T"]), k
        elif T_tol is not None:
            assert np.abs(o["T"] - r["T"]).max() < T_tol * max(1.0, c["unit"]), k
    return recs


@pytest.mark.parametrize("mode", [R.PLANE, R.POINT, R.COLORED], ids=["plane", "point", "colored"])
@pytest.mark.parametrize("n", [1, 257, 8193])
def test_surface(oracle, mode, n):
    # n = 1: one match.  Point-to-plane (rank 1, rejected by both solvers) and point-to-point (zero cross-covariance)
    # stay at init bit for bit; coloured has a rank-2 system whose solution is rounding residue, so pass 0 only
    if n == 1 and mode == R.COLORED:
        check(oracle, IC.surface_pair(n, seed=n), mode, ks=(0,))
    else:
        check(oracle, IC.surface_pair(n, seed=n), mode, exact_T=n == 1)


@pytest.mark.parametrize("unit", [1.0, 1000.0], ids=["m", "mm"])
def test_far_from_the_origin(oracle, unit):
    c = IC.surface_pair(30000, seed=17, unit=unit, offset=1e4 * unit)
    c["init"] = IC.about(IC.rot(1e-4, -2e-4, 1.5e-4), np.full(3, 1e4 * unit), np.array([3e-3, -2e-3, 1e-3]) * unit)
    check(oracle, c, ks=(0,), exact_T=True)


def test_gate_faces_edges_corners(oracle):
    c = IC.gate_case()
    recs = check(oracle, c)
    # the construction: of every four sources beyond a face / edge / corner, the one an ulp inside and the one
    # halfway are matched, the one exactly at the gate and the one beyond it are not; the far points never are
    p = recs[0]["partner"]
    d2 = R.d2_exact(c["src"].astype(np.float64), c["tgt"][np.maximum(p, 0)].astype(np.float64))
    assert recs[0]["ncorr"] == 2 * 26 and (d2[p >= 0] < 225.0).all() and d2[p >= 0].max() > 225.0 - 1e-4


def test_one_point_target(oracle):
    c = IC.one_point_target()
    recs = check(oracle, c, ks=(0,), exact_T=True)
    assert list(np.flatnonzero(recs[0]["partner"] >= 0)) == [1, 2]


def test_ties_go_to_the_lower_index(oracle):
    c = IC.ties_case()
    recs = check(oracle, c)
    # brute force over every target row: the lowest index among the rows at the minimal d²
    s, t = c["src"].astype(np.float64), c["tgt"].astype(np.float64)
    d2 = R.d2_exact(s[:, None, :], t[None, :, :])
    d2 = np.where(d2 < c["max_corr"] ** 2, d2, np.inf)
    lo = np.where(d2 == d2.min(1, keepdims=True), np.arange(len(t))[None, :], len(t)).min(1)
    assert np.array_equal(recs[0]["partner"], np.where(np.isfinite(d2.min(1)), lo, -1))
    assert (np.sum(d2 == d2.min(1, keepdims=True), 1) >= 2).all()        # every source sees a tie of at least two rows


def test_nan_rows_are_absent_but_counted(oracle):
    c = IC.nan_case()
    recs = check(oracle, c)
    assert recs[0]["fitness"] == recs[0]["ncorr"] / len(c["src"]) and (recs[0]["partner"][::7] == -1).all()
    assert not np.isin(recs[0]["partner"], np.arange(5, len(c["tgt"]), 11)).any()


@pytest.mark.parametrize("which", ["all_nan", "empty_src", "empty_tgt"])
def test_nothing_to_match(oracle, which):
    c = IC.surface_pair(300, seed=4)
    c["init"] = IC.rot(0.1, -0.2, 0.3)
    c["init"][:3, 3] = (0.01, 0.02, -0.03)
    if which == "all_nan":
        c["src"][:] = np.nan
    elif which == "empty_src":
        c["src"] = c["src"][:0]
    else:
        c["tgt"], c["tgt_n"] = c["tgt"][:0], c["tgt_n"][:0]
    recs = check(oracle, c, exact_T=True)
    assert all(r["ncorr"] == 0 and r["fitness"] == 0.0 and np.array_equal(r["T"], c["init"]) for r in recs)


def test_planar_zero_residual_keeps_init(oracle):
    recs = check(oracle, IC.planar_case(), exact_T=True)
    assert all(np.array_equal(r["T"], np.eye(4)) and not r["b"].any() for r in recs)


@pytest.mark.parametrize("mode", [R.PLANE, R.POINT, R.COLORED], ids=["plane", "point", "colored"])
@pytest.mark.parametrize("nmatch", [1, 2])
def test_one_and_two_matches(oracle, mode, nmatch):
    c = IC.few_matches_case(nmatch)
    one = nmatch == 1 and mode != R.COLORED
    recs = check(oracle, c, mode, exact_T=True) if one else check(oracle, c, mode, ks=(0,))
    assert recs[0]["ncorr"] == nmatch


@pytest.mark.parametrize("axis_aligned", [True, False], ids=["axis", "general"])
def test_collinear_point_to_point(oracle, axis_aligned):
    c = IC.collinear_case(axis_aligned)
    recs = check(oracle, c, R.POINT, T_tol=None, rmse_abs=1e-8)
    s = c["src"].astype(np.float64)
    for k in KS:
        o = oracle_run(oracle, c, R.POINT, k)
        assert np.abs(R.affine(o["T"], s) - R.affine(recs[k]["T"], s)).max() < 1e-6
        assert abs(np.linalg.det(o["T"][:3, :3]) - 1) < 1e-12


def test_coplanar_point_to_point_is_a_rotation(oracle):
    c = IC.coplanar_reflection_case()
    recs = check(oracle, c, R.POINT)
    assert all(abs(np.linalg.det(r["T"][:3, :3]) - 1) < 1e-12 for r in recs)


def test_stop_rule(oracle):
    c = IC.surface_pair(3000, seed=8)
    recs, res = R.icp(c["src"], c["tgt"], c["max_corr"], tgt_normals=c["tgt_n"])
    o = oracle.icp_point_to_plane(c["src"], c["tgt"], c["tgt_n"], c["max_corr"])
    assert 2 <= res["iters"] < 30 and o["iters"] == res["iters"] and o["ncorr"] == res["ncorr"]
    assert np.abs(o["T"] - res["T"]).max() < 1e-9
