"""CPU reference of the frame engine's floor stage with its reported plane (``floor_mode``, ``floor_plane``), composed
from the oracle's pinned pieces, which it uses unchanged.  Test infrastructure, like the oracle: imported by ``tests/``
only.

Everything up to the filter output (the SOR output, or the radius filter's survivors) and the ICP branch come from
``tests/ror_oracle.py`` / ``tests/c5_oracle.py`` run without the floor stage (their cloud is then the filter output).
The floor stage is restated on that output:

* RANSAC mode (``FLOOR_RANSAC``, the default): band, ``oracle.ransac_plane``, merge and floor SOR with the oracle's rules
  (DESIGN §6), and the frame's plane is ``ransac_plane``'s refit plane, NaN x 4 where the frame has none;
  ``tests/test_oracle_floor_rules.py`` checks that it reproduces ``oracle.frame_pipeline`` (cloud, counts, ``plane``).
* plane mode (``FLOOR_PLANE``): ``oracle.plane_side`` (pcd_above_plane) on the filter output, then ``_sor_or_all``; no
  floor-skip rule, and the reported plane is the caller's.

The crop and the fixed-N slot compose as in ``tests/c5_oracle.py``."""
import types

import numpy as np

import c5_oracle
import ror_oracle

FLOOR_RANSAC, FLOOR_PLANE = 0, 1
NAN4 = np.full(4, np.nan)


def floor_stage(orc, cfg, A):
    """The floor stage on the filter output ``A``: (points, n_floor_inliers, stages, plane)."""
    st = {"n_lo": 0, "n_rest": 0, "n_merged": 0, "n_fsor": 0}
    if not cfg.do_floor:
        return A, 0, st, NAN4.copy()
    if getattr(cfg, "floor_mode", FLOOR_RANSAC) == FLOOR_PLANE:
        a, b, c, d = (float(x) for x in cfg.floor_plane)
        merged = A[orc.plane_side(A, a, b, c, d).astype(bool)] if len(A) else A
        fin = orc._sor_or_all(merged, cfg.floor_sor_k, cfg.floor_sor_ratio) if len(merged) else merged
        st.update(n_merged=len(merged), n_fsor=len(fin) if cfg.floor_sor_k > 0 else 0)
        return fin, len(A) - len(merged), st, np.array([a, b, c, d], np.float64)
    if len(A) == 0:
        return A, 0, st, NAN4.copy()
    low = orc.band_mask(A, cfg.floor_band, 1).astype(bool)
    floor, upper = A[low], A[~low]
    if len(floor) >= cfg.ransac_n:
        plane, inl, _, _ = orc.ransac_plane(floor, cfg.ransac_thr, cfg.ransac_n, cfg.ransac_iters, seed=cfg.seed)
        inl = inl.astype(bool)
    else:                                   # no hypothesis can be drawn: no plane, nobody is an inlier
        plane, inl = NAN4.copy(), np.zeros(len(floor), bool)
    merged = np.concatenate([floor[~inl], upper], 0)
    fin = orc._sor_or_all(merged, cfg.floor_sor_k, cfg.floor_sor_ratio)
    st.update(n_lo=len(floor), n_rest=len(floor) - int(inl.sum()), n_merged=len(merged),
              n_fsor=len(fin) if cfg.floor_sor_k > 0 else 0)
    if len(A) < cfg.ransac_n:               # floor stage skipped: the filter output stays the frame's cloud
        return A, 0, st, NAN4.copy()
    return fin, int(inl.sum()), st, np.asarray(plane, np.float64)


def frame_pipeline(orc, cfg, depth_f, tab, T_fuse, T_icp, want_icp=True, stages=False, rgb_f=None, frame_id=0):
    """The engine's frame composition with the floor stage in either mode, the radius filter, the crop and the fixed-N
    slot.  Adds ``floor_plane`` (float64 [4]) to the result."""
    plain = types.SimpleNamespace(**dict(vars(cfg), do_floor=False, resample_n=0))
    base = ror_oracle.frame_pipeline(orc, plain, depth_f, tab, T_fuse, T_icp, want_icp=want_icp, stages=True, rgb_f=rgb_f)
    pts, ninl, st, plane = floor_stage(orc, cfg, base["points"])
    out = {k: base[k] for k in ("n_fused", "n_voxel", "n_sor", "icp")}
    out.update(points=pts, n_floor_inliers=ninl, floor_plane=plane)
    if "crop_median" in base:
        out["crop_median"] = base["crop_median"]
    if stages:
        out.update(st, n_ror=base["n_ror"], nv_icp=base["nv_icp"], n_icp=base["n_icp"])
    if getattr(cfg, "resample_n", 0) > 0:
        out["fixed"], out["fixed_status"] = c5_oracle.fixed_slot(orc, pts, cfg.resample_n, cfg.resample_mode, cfg.seed, frame_id)
    return out
