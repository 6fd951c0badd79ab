"""CPU reference of the frame engine's config C5 rules -- the human crop and the fixed-N slot -- composed from the
oracle's pinned pieces (``oracle.crop_mask``, ``oracle.frame_pipeline``, ``oracle.resample_fixed_n``), which it uses
unchanged.  Test infrastructure, like the oracle: imported by ``tests/`` only.

The crop (preprocessing/data.py:165-178) removes pixels from the fused cloud.  A pixel with depth 0 is invalid in the
unprojection whatever the flags, so the cropped fused cloud is exactly the oracle's composition run on a depth image
whose cropped pixels are set to 0.  The ICP branch registers the uncropped clouds, as the reference does
(data.py:140-142), so its results are those of the oracle's composition on the original depth."""
import numpy as np


def crop_z16(depth_s, tab_s):
    """The int16 z column of one sensor's `_depth.dat` as the crop reads it: (int16)depth, 0 outside the table (so a
    depth >= 32768 is negative)."""
    tab_s = np.asarray(tab_s, dtype=np.float32).reshape(-1, 2)
    out = np.asarray(depth_s, dtype=np.uint16).reshape(-1).astype(np.int16)
    out[np.isnan(tab_s[:, 0]) | np.isnan(tab_s[:, 1])] = 0
    return out


def frame_crop(orc, rgb_f, depth_f, tab, gate):
    """The crop of every sensor of a frame through ``oracle.crop_mask`` (numpy's median over all P z values): the keep
    mask [S*P] and the per-sensor medians."""
    keeps, meds = [], []
    for s in range(depth_f.shape[0]):
        z = crop_z16(depth_f[s], tab[s])
        k, m = orc.crop_mask(np.asarray(rgb_f[s]).reshape(-1, 3), np.stack([np.zeros_like(z), np.zeros_like(z), z], 1), gate)
        keeps.append(k.astype(bool))
        meds.append(m)
    return np.concatenate(keeps), meds


def fixed_slot(orc, points, N, mode, seed, frame_id):
    """One frame's fixed-N slot: ``resample_fixed_n`` with stream = frame id; PREFIX (mode 1) zero-pads a short cloud;
    a RANDOM cloud with fewer than N points gives (zeros, KP_E_ARG = -1)."""
    slot = np.zeros((int(N), 3), np.float32)
    try:
        got, _ = orc.resample_fixed_n(points, N, "prefix" if mode == 1 else "random", seed=seed, stream=frame_id)
    except ValueError:
        return slot, -1
    slot[:len(got)] = got
    return slot, 0


def frame_pipeline(orc, cfg, depth_f, tab, T_fuse, T_icp, want_icp=True, stages=False, rgb_f=None, frame_id=0):
    """``oracle.frame_pipeline`` with the engine's crop (``cfg.do_crop``, ``rgb_f`` uint8 [S,P,3]: adds
    ``crop_median``) and fixed-N output (``cfg.resample_n`` > 0: adds ``fixed`` [N,3] and ``fixed_status``)."""
    depth_f = np.asarray(depth_f, dtype=np.uint16)
    if not getattr(cfg, "do_crop", False):
        out = orc.frame_pipeline(cfg, depth_f, tab, T_fuse, T_icp, want_icp=want_icp, stages=stages)
    else:
        if rgb_f is None:
            raise ValueError("the crop needs the frame's segmentation images")
        keep, meds = frame_crop(orc, rgb_f, depth_f, tab, cfg.crop_gate)
        cropped = depth_f.copy().reshape(-1)
        cropped[~keep] = 0
        out = orc.frame_pipeline(cfg, cropped.reshape(depth_f.shape), tab, T_fuse, T_icp, want_icp=False, stages=stages)
        out["crop_median"] = meds
        if want_icp and cfg.do_icp and depth_f.shape[0] > 1:
            full = orc.frame_pipeline(cfg, depth_f, tab, T_fuse, T_icp, want_icp=True, stages=True)
            out["icp"] = full["icp"]
            if stages:
                out["nv_icp"], out["n_icp"] = full["nv_icp"], full["n_icp"]
    if getattr(cfg, "resample_n", 0) > 0:
        out["fixed"], out["fixed_status"] = fixed_slot(orc, out["points"], cfg.resample_n, cfg.resample_mode, cfg.seed, frame_id)
    return out
