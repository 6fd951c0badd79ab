"""Float64 reference of one ICP run, pass by pass: the arithmetic contract of DESIGN §3 for registration_icp (point-to-plane,
point-to-point) and registration_colored_icp, restated with NumPy / SciPy only.  Test infrastructure, like the oracle:
imported by ``tests/`` only, and independent of the oracle's ICP.

* Moving source: ``cur = init · src`` in double, per row ``((a·x + b·y) + c·z) + d`` (the order of ``kp_affine``), then
  moved in place by each pass's update U in the same order.  Rows with a NaN coordinate are absent: never matched, but
  counted in n_src for the fitness.
* Partner: among the target rows without NaN, the one with the smallest ``d² = (dx·dx + dy·dy) + dz·dz`` in double on
  the float32-stored target, under the strict gate ``d² < max_corr²``; ties go to the lower target index.  The k-d tree
  only collects candidates (with a margin); the decision is taken in that expression.
* Per-pass sums: point-to-plane ``J = [s × n, n]``, ``r = (s − t)·n``; coloured: √λ times that row plus √(1−λ) times
  the photometric row of ``icp_tile_terms`` (target gradient supplied by the caller, as ``kp_color_gradient`` computes
  it); point-to-point: Umeyama by a NumPy SVD with the det correction, identity for a zero cross-covariance.
* Update: the 6×6 by ``numpy.linalg.solve`` (identity when there is no match or the system is singular or its solution
  not finite), U = (Rz Ry Rx | t), T ← U·T.
* Stop rule (Open3D's): after pass k > 0, stop when |Δfitness| < rel_fit and |Δrmse| < rel_rmse, or at k = max_iter.

``passes`` yields, for every pass k, the state after it: ncorr, fitness, rmse, T (after k updates: what the kernels
report for ``max_iter = k``), the partner of every source row (-1 = none) and, for the 6×6 modes, the system."""
import math

import numpy as np
from scipy.spatial import cKDTree

PLANE, POINT, COLORED = 0, 1, 2


def affine(T, P):
    """Rows of P moved by the 3x4 part of T, each coordinate ((a·x + b·y) + c·z) + d (no contraction: NumPy ufuncs)."""
    x, y, z = P[:, 0], P[:, 1], P[:, 2]
    return np.stack([((T[i, 0] * x + T[i, 1] * y) + T[i, 2] * z) + T[i, 3] for i in range(3)], axis=1)


def d2_exact(s, t):
    e = s - t
    return (e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2]


class Partners:
    """Exact nearest target row inside the gate, canonical (d², index) order."""
    K = 4                      # candidates fetched per query; a tie set that may reach past them is re-collected whole

    def __init__(self, tgt, max_corr):
        self.t64 = np.asarray(tgt, np.float32).reshape(-1, 3).astype(np.float64)
        self.ids = np.flatnonzero(~np.isnan(self.t64).any(1))
        self.tree = cKDTree(self.t64[self.ids]) if len(self.ids) else None
        self.max_corr, self.r2 = float(max_corr), float(max_corr) * float(max_corr)

    def _decide(self, q, cand):
        """Best original index among candidate rows `cand` (original indices) for query q, or -1."""
        if len(cand) == 0:
            return -1
        cand = np.asarray(cand, np.int64)
        d2 = d2_exact(q[None, :], self.t64[cand])
        ok = d2 < self.r2
        if not ok.any():
            return -1
        d2, cand = d2[ok], cand[ok]
        return int(cand[d2 == d2.min()].min())

    def __call__(self, cur):
        n = len(cur)
        out = np.full(n, -1, np.int64)
        live = np.flatnonzero(~np.isnan(cur).any(1))
        if self.tree is None or len(live) == 0:
            return out
        q = cur[live]
        K = min(self.K, len(self.ids))
        dist, j = self.tree.query(q, k=K, distance_upper_bound=self.max_corr * (1 + 1e-6), workers=-1)
        dist, j = dist.reshape(len(q), K), j.reshape(len(q), K)
        valid = j < len(self.ids)
        cand = self.ids[np.where(valid, j, 0)]
        d2 = np.where(valid, d2_exact(q[:, None, :], self.t64[cand]), np.inf)
        d2 = np.where(d2 < self.r2, d2, np.inf)
        best = d2.min(1)
        big = np.iinfo(np.int64).max
        pick = np.where((d2 == best[:, None]) & np.isfinite(d2), cand, big).min(1)
        has = np.isfinite(best)
        res = np.where(has, pick, -1)
        # the tree's distances are not the decision's: where its K-th candidate is within a relative 1e-9 of the best,
        # a point it did not return could tie with or beat the best, so that query is decided over its whole ball
        # (with best = inf: K candidates near the gate all failed it, and one the tree ranked behind them may pass)
        redo = valid[:, K - 1] & (dist[:, K - 1] ** 2 <= np.minimum(best, self.r2) * (1 + 1e-9))
        for r in np.flatnonzero(redo):
            ball = self.tree.query_ball_point(q[r], math.sqrt(min(best[r], self.r2)) * (1 + 1e-8) + 1e-300)
            res[r] = self._decide(q[r], self.ids[np.asarray(ball, np.int64)])
        out[live] = res
        return out


def x6_to_mat4(x):
    """U = (Rz(x2) Ry(x1) Rx(x0) | x3..5)."""
    ca, sa, cb, sb, cg, sg = math.cos(x[0]), math.sin(x[0]), math.cos(x[1]), math.sin(x[1]), math.cos(x[2]), math.sin(x[2])
    Rx = np.array([[1, 0, 0], [0, ca, -sa], [0, sa, ca]])
    Ry = np.array([[cb, 0, sb], [0, 1, 0], [-sb, 0, cb]])
    Rz = np.array([[cg, -sg, 0], [sg, cg, 0], [0, 0, 1]])
    U = np.eye(4)
    U[:3, :3] = Rz @ Ry @ Rx
    U[:3, 3] = x[3:6]
    return U


def umeyama(s, t):
    """Eigen::umeyama without scaling on matched rows: R = U diag(1, 1, det U det V) Vᵀ of the cross-covariance
    (1/n) Σ (t − mt)(s − ms)ᵀ, translation mt − R ms; identity when the cross-covariance vanishes."""
    U4 = np.eye(4)
    if len(s) == 0:
        return U4
    ms, mt = s.mean(0), t.mean(0)
    C = (t - mt).T @ (s - ms) / len(s)
    u, S, vt = np.linalg.svd(C)
    if not S[0] > 1e-300:
        return U4
    d = -1.0 if np.linalg.det(u) * np.linalg.det(vt) < 0 else 1.0
    R = u @ np.diag([1.0, 1.0, d]) @ vt
    U4[:3, :3] = R
    U4[:3, 3] = mt - R @ ms
    return U4


def intensity(colors):
    """(r + g + b) / 3 in double on the float32-stored colours, rounded once to float32."""
    c = np.asarray(colors, np.float32).astype(np.float64)
    return (((c[:, 0] + c[:, 1]) + c[:, 2]) / 3.0).astype(np.float32)


def _system(mode, s, t, n, lam, si, ti, tg):
    """JᵀJ, Jᵀr of the matched rows (point-to-plane / coloured)."""
    e = s - t
    r = (e[:, 0] * n[:, 0] + e[:, 1] * n[:, 1]) + e[:, 2] * n[:, 2]
    J = np.stack([s[:, 1] * n[:, 2] - s[:, 2] * n[:, 1], s[:, 2] * n[:, 0] - s[:, 0] * n[:, 2],
                  s[:, 0] * n[:, 1] - s[:, 1] * n[:, 0], n[:, 0], n[:, 1], n[:, 2]], axis=1)
    if mode != COLORED:
        return J.T @ J, J.T @ r
    slg, slp = math.sqrt(lam), math.sqrt(1.0 - lam)
    p = e - r[:, None] * n                                      # vs_proj - vt
    is_proj = ((tg[:, 0] * p[:, 0] + tg[:, 1] * p[:, 1]) + tg[:, 2] * p[:, 2]) + ti
    gn = (tg[:, 0] * n[:, 0] + tg[:, 1] * n[:, 1]) + tg[:, 2] * n[:, 2]
    m = -(tg - gn[:, None] * n)                                 # -(I - n nᵀ) grad
    J2 = slp * np.stack([s[:, 1] * m[:, 2] - s[:, 2] * m[:, 1], s[:, 2] * m[:, 0] - s[:, 0] * m[:, 2],
                         s[:, 0] * m[:, 1] - s[:, 1] * m[:, 0], m[:, 0], m[:, 1], m[:, 2]], axis=1)
    r2 = slp * (si - is_proj)
    J, r = slg * J, slg * r
    return J.T @ J + J2.T @ J2, J.T @ r + J2.T @ r2


def passes(src, tgt, max_corr, init=None, mode=PLANE, tgt_normals=None, src_colors=None, tgt_colors=None, tgt_grad=None,
           lam=0.968):
    """Generator over the passes of an ICP run that never stops: pass k's dict (see the module docstring)."""
    src = np.asarray(src, np.float32).reshape(-1, 3)
    tgt = np.asarray(tgt, np.float32).reshape(-1, 3)
    T = np.array(np.eye(4) if init is None else init, np.float64)
    cur = affine(T, src.astype(np.float64))
    find = Partners(tgt, max_corr)
    t64 = find.t64
    n64 = None if tgt_normals is None else np.asarray(tgt_normals, np.float32).reshape(-1, 3).astype(np.float64)
    si = ti = tg = None
    if mode == COLORED:
        si = intensity(src_colors).astype(np.float64)
        ti = intensity(tgt_colors).astype(np.float64)
        tg = np.asarray(tgt_grad, np.float32).reshape(-1, 3).astype(np.float64)
    ns = len(src)
    k = 0
    while True:
        p = find(cur)
        m = np.flatnonzero(p >= 0)
        j = p[m]
        s, t = cur[m], t64[j]
        nc = len(m)
        err2 = math.fsum(d2_exact(s, t))
        rec = {"pass": k, "ncorr": nc, "fitness": nc / ns if ns else 0.0, "rmse": math.sqrt(err2 / nc) if nc else 0.0,
               "T": T.copy(), "partner": p, "A": None, "b": None}
        U = np.eye(4)
        if mode == POINT:
            U = umeyama(s, t)
        elif nc:
            A, b = _system(mode, s, t, n64[j], lam, None if si is None else si[m], None if ti is None else ti[j],
                           None if tg is None else tg[j])
            rec["A"], rec["b"] = A, b
            try:
                x = np.linalg.solve(A, -b)
                if np.isfinite(x).all():
                    U = x6_to_mat4(x)
            except np.linalg.LinAlgError:
                pass
        yield rec
        T = U @ T
        cur = affine(U, cur)
        k += 1


def icp(src, tgt, max_corr, init=None, max_iter=30, rel_fit=1e-6, rel_rmse=1e-6, **kw):
    """A whole run with Open3D's stop rule: (list of pass records, result dict shaped like the oracle's)."""
    out = []
    for rec in passes(src, tgt, max_corr, init=init, **kw):
        out.append(rec)
        k = rec["pass"]
        if k > 0 and abs(out[-2]["fitness"] - rec["fitness"]) < rel_fit and abs(out[-2]["rmse"] - rec["rmse"]) < rel_rmse:
            break
        if k >= max_iter:
            break
    last = out[-1]
    res = {"T": last["T"], "fitness": last["fitness"], "rmse": last["rmse"], "iters": last["pass"], "ncorr": last["ncorr"]}
    return out, res
