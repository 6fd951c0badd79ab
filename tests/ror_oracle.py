"""CPU reference of the frame engine's radius outlier removal (``ror_nb_points``, ``ror_radius``), composed from the
oracle's pinned pieces, which it uses unchanged.  Test infrastructure, like the oracle: imported by ``tests/`` only.

The stage filters ``A``, the SOR output (the voxel output when ``sor_k = 0``), with ``oracle.radius_outlier``, and its
survivors replace ``A`` downstream.  Everything up to ``A`` and the ICP branch, which never sees the stage, is
``oracle.frame_pipeline`` run without the floor stage (its cloud is then ``A``).  The floor stage is restated on the
survivors with the oracle's rules (DESIGN §6); ``floor_stage`` on ``A`` itself reproduces ``oracle.frame_pipeline``, which
``tests/test_oracle_ror_rules.py`` checks.  The crop and the fixed-N slot compose as in ``tests/c5_oracle.py``."""
import types

import numpy as np

import c5_oracle


def floor_stage(orc, cfg, A):
    """The floor stage of ``oracle.frame_pipeline`` on the filter output ``A``: (points, n_floor_inliers, stages)."""
    st = {"n_lo": 0, "n_rest": 0, "n_merged": 0, "n_fsor": 0}
    if not cfg.do_floor or len(A) == 0:
        return A, 0, st
    low = orc.band_mask(A, cfg.floor_band, 1).astype(bool)
    floor, upper = A[low], A[~low]
    if len(floor) >= cfg.ransac_n:
        _, inl, _, _ = orc.ransac_plane(floor, cfg.ransac_thr, cfg.ransac_n, cfg.ransac_iters, seed=cfg.seed)
        inl = inl.astype(bool)
    else:                                   # no hypothesis can be drawn: nobody is an inlier
        inl = np.zeros(len(floor), bool)
    merged = np.concatenate([floor[~inl], upper], 0)
    fin = orc._sor_or_all(merged, cfg.floor_sor_k, cfg.floor_sor_ratio)
    st.update(n_lo=len(floor), n_rest=len(floor) - int(inl.sum()), n_merged=len(merged),
              n_fsor=len(fin) if cfg.floor_sor_k > 0 else 0)
    if len(A) < cfg.ransac_n:               # floor stage skipped: the filter output stays the frame's cloud
        return A, 0, st
    return fin, int(inl.sum()), st


def frame_pipeline(orc, cfg, depth_f, tab, T_fuse, T_icp, want_icp=True, stages=False, rgb_f=None, frame_id=0):
    """The engine's frame composition with the radius filter (``cfg.ror_nb_points`` > 0), the crop (``cfg.do_crop``,
    ``rgb_f``) and the fixed-N slot (``cfg.resample_n`` > 0).  ``stages=True`` adds ``n_ror`` (0 when the stage is off)."""
    nb = getattr(cfg, "ror_nb_points", 0)
    if nb <= 0:
        out = c5_oracle.frame_pipeline(orc, cfg, depth_f, tab, T_fuse, T_icp, want_icp=want_icp, stages=stages, rgb_f=rgb_f,
                                       frame_id=frame_id)
        if stages:
            out["n_ror"] = 0
        return out
    # up to the filter output, and ICP: the oracle's composition without the floor stage (its cloud is then A)
    plain = types.SimpleNamespace(**dict(vars(cfg), do_floor=False, resample_n=0))
    base = c5_oracle.frame_pipeline(orc, plain, depth_f, tab, T_fuse, T_icp, want_icp=want_icp, stages=True, rgb_f=rgb_f)
    A = base["points"]
    R = A[orc.radius_outlier(A, nb, cfg.ror_radius)[0].astype(bool)] if len(A) else A
    pts, ninl, st = floor_stage(orc, cfg, R)
    out = {k: base[k] for k in ("n_fused", "n_voxel", "n_sor", "icp")}
    out.update(points=pts, n_floor_inliers=ninl)
    if "crop_median" in base:
        out["crop_median"] = base["crop_median"]
    if stages:
        out.update(st, n_ror=len(R), nv_icp=base["nv_icp"], n_icp=base["n_icp"])
    if getattr(cfg, "resample_n", 0) > 0:
        out["fixed"], out["fixed_status"] = c5_oracle.fixed_slot(orc, pts, cfg.resample_n, cfg.resample_mode, cfg.seed, frame_id)
    return out
