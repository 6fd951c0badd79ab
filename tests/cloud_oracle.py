"""CPU reference of the frame engine's cloud input (``input_mode = INPUT_CLOUDS``), composed from the oracle's pinned
pieces, which it uses unchanged.  Test infrastructure, like the oracle: imported by ``tests/`` only.

A saved cloud enters the engine's stages from the voxel downsample on: its rows with x NaN are dropped (the others keep
their order), then ``oracle.voxel_downsample`` when ``cloud_voxel = 1``, ``oracle._sor_or_all``, ``oracle.radius_outlier``
(composed as ``tests/ror_oracle.py`` composes it), ``floor_oracle.floor_stage`` and ``c5_oracle.fixed_slot``.
``tests/test_oracle_cloud_rules.py`` holds the composition to ``oracle.remove_floor`` (the ``floor_removal.py`` body) and
``oracle.filter_outliers``.  ``fused_clouds`` makes the synthetic inputs: the fused clouds of rendered frames, as the
reference's ``DataProcessor`` saved them."""
import numpy as np

from kinectpy_b200 import synth

import c5_oracle
import floor_oracle

SMALL = synth.SensorMode("SMALL", 160, 120, 126.0, 126.0, 79.5, 59.5, "hexagon")


def fused_clouds(orc, frames=1, first=0, mode=SMALL, S=3, voxel_mm=10.0):
    """Fused clouds in millimetres of ``frames`` rendered frames: every sensor's unprojection through its extrinsic, the
    valid rows voxel-downsampled at ``voxel_mm`` (the saved clouds are filter outputs), float32 [n, 3] each."""
    depth, tab, T = synth.render_sequence(mode, frames, S, first_frame=first)
    Tmm = synth.scale_extrinsics(T, 1.0)
    out = []
    for f in range(frames):
        xyz, valid, _ = orc.unproject(depth[f][None], tab, Tmm, flags=orc.F_INT16 | orc.F_DROP_ANY_ZERO, scale=1.0)
        rows = xyz[0][valid[0].astype(bool)]
        out.append(np.ascontiguousarray(orc.voxel_downsample(rows, voxel_mm)["points"], np.float32))
    return out


def cloud_pipeline(orc, cfg, pts, frame_id=0):
    """One cloud through the engine's stages: the result record's counts, the final cloud (``points``), ``floor_plane``,
    the floor stage's counts (``n_lo`` ... ``n_fsor``), ``n_ror`` and, with ``cfg.resample_n`` > 0, ``fixed`` and
    ``fixed_status``."""
    pts = np.ascontiguousarray(pts, np.float32).reshape(-1, 3)
    rows = pts[~np.isnan(pts[:, 0])]
    out = {"n_fused": len(rows)}
    V = orc.voxel_downsample(rows, cfg.voxel_size)["points"] if cfg.cloud_voxel and len(rows) else rows
    out["n_voxel"] = len(V)
    A = orc._sor_or_all(V, cfg.sor_k, cfg.sor_ratio) if len(V) else V
    out["n_sor"] = len(A)
    nb = cfg.ror_nb_points
    R = A[orc.radius_outlier(A, nb, cfg.ror_radius)[0].astype(bool)] if nb > 0 and len(A) else A
    fin, ninl, st, plane = floor_oracle.floor_stage(orc, cfg, R)
    out.update(st, points=fin, n_floor_inliers=ninl, floor_plane=plane, n_ror=len(R) if nb > 0 else 0)
    if cfg.resample_n > 0:
        out["fixed"], out["fixed_status"] = c5_oracle.fixed_slot(orc, fin, cfg.resample_n, cfg.resample_mode, cfg.seed, frame_id)
    return out


def cloud_cfg(P, **kw):
    """A cloud-input PipelineConfig; the defaults are ``floor_removal.py``'s body in millimetres: no voxel step, no
    filter SOR, band 200, RANSAC threshold 30 with 30-point hypotheses and 2000 iterations, floor SOR 50 / 0.30 (the
    point spacing, 10 mm, only sizes the neighbour grids)."""
    from kinectpy_b200 import _cabi
    from kinectpy_b200.pipeline import PipelineConfig
    base = dict(input_mode=_cabi.INPUT_CLOUDS, cloud_voxel=0, n_sensors=1, pixels=int(P), scale=1.0, voxel_size=10.0,
                sor_k=0, sor_ratio=2.0, do_floor=True, floor_band=200.0, ransac_thr=30.0, ransac_n=30, ransac_iters=2000,
                floor_sor_k=50, floor_sor_ratio=0.30, do_icp=False, seed=1234, n_streams=1)
    base.update(kw)
    return PipelineConfig(**base)
