"""CPU premise check for the ICP list path (counts only -- no timing; nothing here says anything about B200 speed).

For one synthetic frame of bench.py's C4 workload (WFOV, 3 sensors, ICP start as in bench.py) it runs a NumPy / cKDTree
point-to-plane ICP of both sub clouds against the master's 1 cm voxel cloud and reports, per pass:
  * the share of source points whose previous partner t satisfies  4 * d2(q, t) * (1 + 1e-6) < rho2_L(t),
    where rho2_L(t) is the squared completeness radius of t's hybrid normals list (r = 2 cm, 30 nn) cut to L entries
    besides t itself -- such a point's exact partner is t or one of those L entries (triangle inequality);
  * how many list entries lie within 2 * d(q, t) (what the list path would evaluate);
  * whether the brute-force partner was in the list every time (it must be);
  * at passes 2, 4, 8: how list-path points fall into 32-point warps in the source's voxel order.
Usage: python tools/icp_list_premise.py  (from any directory; needs gcc for the oracle and scipy).
"""
import os
import sys
import time

import numpy as np
from scipy.spatial import cKDTree

REPO = os.environ.get("KP_REPO", os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)
import bench                      # noqa: E402  (make_inputs: the benchmark's own frames, extrinsics and ICP start)
from oracle import oracle as orc  # noqa: E402

R, MAXNN, MAXC, VOX = 0.02, 30, 0.02, 0.01
LS = (4, 8, 12, 29)


def main():
    t0 = time.time()
    orc.build()
    mode, depth, tab, T_fuse, T_icp = bench.make_inputs("WFOV", 1, 0)
    d = depth[0]
    P = mode.pixels
    xyz, _, _ = orc.unproject(d[None], tab, T_fuse, flags=0, scale=1e-3)
    tgt = orc.voxel_downsample(xyz[0][:P], VOX)["points"].astype(np.float64)
    tree = cKDTree(tgt)
    dd, ii = tree.query(tgt, k=MAXNN, distance_upper_bound=R)      # hybrid list, self first, ascending
    dd2, cnt = dd ** 2, np.isfinite(dd).sum(1)
    nrm = orc.estimate_normals(tgt.astype(np.float32), R, MAXNN).astype(np.float64)

    def rho2(L):      # list = self + first L others; complete for d2 < rho2
        r = np.where(cnt < MAXNN, R * R, dd2[:, MAXNN - 1])
        return np.where(cnt > L + 1, dd2[:, min(L + 1, MAXNN - 1)], r)

    RH = {L: rho2(L) for L in LS}
    print("target points %d; median target nn distance %.2f mm; median rho per L (cm): %s" % (
        len(tgt), 1e3 * np.median(dd[:, 1][np.isfinite(dd[:, 1])]),
        {L: round(100 * float(np.sqrt(np.median(RH[L]))), 2) for L in LS}))
    for s in (1, 2):
        raw, _, _ = orc.unproject(d[None, s:s + 1], tab[s:s + 1], None, flags=0, scale=1e-3)
        src = orc.voxel_downsample(raw[0], VOX)["points"].astype(np.float64)
        T = T_icp[s]
        cur = src @ T[:3, :3].T + T[:3, 3]
        prev, pfit, prmse = None, None, None
        for it in range(31):
            dq, iq = tree.query(cur, k=1, distance_upper_bound=MAXC)
            has = np.isfinite(dq)
            if prev is not None:
                pv = prev >= 0
                p0 = np.where(pv, prev, 0)
                delta2 = np.where(pv, ((cur - tgt[p0]) ** 2).sum(1), np.inf)
                okp = pv & (delta2 < MAXC * MAXC)
                share = {L: (okp & (4 * delta2 * (1 + 1e-6) < RH[L][p0])).mean() for L in LS}
                cond = okp & (4 * delta2 * (1 + 1e-6) < RH[12][p0])
                sel = np.where(cond)[0]
                within = (dd2[prev[sel], 1:13] <= (4 * delta2[sel] * (1 + 1e-6))[:, None]).sum(1)
                exact = ((ii[prev[sel], :13] == iq[sel][:, None]).any(1) | ~has[sel]).all()
                print("pair %d pass %2d  matched %.3f  list-path share %s  entries within 2d: mean %.2f p90 %d  partner in list: %s" % (
                    s, it, has.mean(), " ".join("L=%d %.3f" % kv for kv in share.items()), within.mean(),
                    np.percentile(within, 90), bool(exact)))
                if it in (2, 4, 8):
                    n32 = ((len(cur) + 31) // 32) * 32
                    Wl = np.zeros(n32, bool); Wl[:len(cur)] = cond
                    Wg = np.zeros(n32, bool); Wg[:len(cur)] = ~cond
                    Wl, Wg = Wl.reshape(-1, 32), Wg.reshape(-1, 32)
                    mixed = Wl.any(1) & Wg.any(1)
                    print("      warps of 32 (voxel order): all list %.3f, all grid %.3f, mixed %.3f (%.1f grid lanes each)" % (
                        (~Wg.any(1)).mean(), (~Wl.any(1)).mean(), mixed.mean(), Wg[mixed].sum(1).mean()))
            m = has
            q, t, n = cur[m], tgt[iq[m]], nrm[iq[m]]
            fit, rmse = m.mean(), np.sqrt((dq[m] ** 2).mean())
            if pfit is not None and abs(pfit - fit) < 1e-6 and abs(prmse - rmse) < 1e-6:
                print("pair %d converged at pass %d" % (s, it))
                break
            pfit, prmse = fit, rmse
            J = np.hstack([np.cross(q, n), n])
            x = np.linalg.solve(J.T @ J, -J.T @ ((q - t) * n).sum(1))
            ca, sa, cb, sb, cg, sg = np.cos(x[0]), np.sin(x[0]), np.cos(x[1]), np.sin(x[1]), np.cos(x[2]), np.sin(x[2])
            U = np.array([[cg * cb, cg * sb * sa - sg * ca, cg * sb * ca + sg * sa],
                          [sg * cb, sg * sb * sa + cg * ca, sg * sb * ca - cg * sa],
                          [-sb, cb * sa, cb * ca]])
            cur = cur @ U.T + x[3:]
            prev = np.where(has, iq, -1)
    print("%.1f s" % (time.time() - t0))


if __name__ == "__main__":
    main()
