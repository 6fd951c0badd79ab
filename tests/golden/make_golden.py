#!/usr/bin/env python
"""Generate tests/golden/reference_own_arithmetic.npz by RUNNING THE REFERENCE'S OWN CODE
(a checkout of tiborcamargo/KinectPy, read-only).

The reference's geometric heavy lifting is Open3D (absent here), but a few steps of the path are
the reference's own numpy arithmetic.  Those are executed here, unmodified, with a minimal
``open3d`` stand-in that only provides containers (PointCloud with points/colors, Vector3dVector,
select_by_index with Open3D's mask-walk order) -- no geometry is computed by the stand-in:

* ``floor_removal.equation_plane`` / ``pcd_above_plane``          (floor_removal.py:21-51)
* ``utils.io.load_depth`` / ``rgbd_to_pointcloud``                  (utils/io.py:15-43)
* ``DataProcessor._transform_filtered_image_to_pointcloud``         (preprocessing/data.py:165-178)
* ``preprocessing.filtering.kalman_filter``                         (preprocessing/filtering.py:98-129)
* the floor-band split expression of the script body                (floor_removal.py:64-66, evaluated verbatim)

Run:  python tests/golden/make_golden.py <KinectPy checkout>        (the .npz is committed)
"""
import contextlib
import io
import os
import sys
import tempfile
import types

import numpy as np

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_own_arithmetic.npz")


def install_stubs():
    class StubPointCloud:
        def __init__(self):
            self.points = np.zeros((0, 3))
            self.colors = np.zeros((0, 3))

        def select_by_index(self, indices, invert=False):
            idx = np.asarray(indices, dtype=np.int64).reshape(-1)
            mask = np.zeros(len(self.points), dtype=bool)
            mask[idx] = True
            if invert:
                mask = ~mask
            out = StubPointCloud()
            out.points = np.asarray(self.points)[mask]
            if len(self.colors) == len(self.points):
                out.colors = np.asarray(self.colors)[mask]
            return out

    o3d = types.ModuleType("open3d")
    o3d.geometry = types.SimpleNamespace(PointCloud=StubPointCloud)
    o3d.utility = types.SimpleNamespace(Vector3dVector=lambda a: np.asarray(a, dtype=np.float64))
    o3d.pipelines = types.SimpleNamespace(registration=types.SimpleNamespace())
    o3d.visualization = types.SimpleNamespace()
    o3d.io = types.SimpleNamespace()
    sys.modules["open3d"] = o3d
    for name in ("tensorflow", "imghdr", "PIL", "PIL.Image"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["PIL"].Image = sys.modules["PIL.Image"]
    return StubPointCloud


def main():
    ref = sys.argv[1]          # a checkout of tiborcamargo/KinectPy
    StubPointCloud = install_stubs()
    sys.path.insert(0, ref)
    import floor_removal as ref_floor
    from preprocessing import filtering as ref_filtering
    from preprocessing.data import DataProcessor
    from utils import io as ref_io

    r = np.random.default_rng(1234)
    out = {}

    # ---- equation_plane (prints; silence it)
    tri = r.normal(size=(16, 3, 3)) * 1000.0
    planes = []
    with contextlib.redirect_stdout(io.StringIO()):
        for t in tri:
            planes.append(ref_floor.equation_plane(t[0], t[1], t[2]))
    out["plane_triples"] = tri
    out["plane_abcd"] = np.array(planes, dtype=np.float64)

    # ---- pcd_above_plane
    cloud = (r.normal(size=(600, 3)) * 800.0).astype(np.float32).astype(np.float64)
    pcd = StubPointCloud()
    pcd.points = cloud
    a, b, c, d = planes[0]
    above = ref_floor.pcd_above_plane(a, b, c, d, pcd)
    out["above_cloud"] = cloud
    out["above_plane"] = np.array([a, b, c, d])
    out["above_points"] = np.asarray(above.points)

    # ---- load_depth / rgbd_to_pointcloud
    n = 48 * 40
    xyz16 = r.integers(-3000, 5000, (n, 3)).astype(np.int16)
    xyz16[r.random(n) < 0.2] = 0
    xyz16[r.random(n) < 0.05, 0] = 0
    xyz16[r.random(n) < 0.05, 1] = 0
    rgb = r.integers(0, 256, (40, 48, 3)).astype(np.uint8)
    with tempfile.TemporaryDirectory() as tmp:
        fp = os.path.join(tmp, "123456")
        xyz16.tofile(fp + "_depth.dat")
        loaded = ref_io.load_depth(fp)
    assert np.array_equal(loaded, xyz16)
    out["dat_xyz16"] = xyz16
    out["dat_rgb"] = rgb
    p = ref_io.rgbd_to_pointcloud(rgb, loaded)
    out["rgbd_points"] = np.asarray(p.points)
    out["rgbd_colors"] = np.asarray(p.colors)

    # ---- human crop (median + 750 gate, non-black pixels), then rgbd_to_pointcloud
    filt = rgb.copy()
    filt[r.random((40, 48)) < 0.55] = 0
    crop = DataProcessor._transform_filtered_image_to_pointcloud(None, filt, loaded)
    out["crop_filtered_img"] = filt
    out["crop_points"] = np.asarray(crop.points)
    out["crop_colors"] = np.asarray(crop.colors)
    out["crop_median"] = np.array(np.median(loaded[:, 2]))

    # ---- floor band expression of floor_removal.py:64-66, evaluated verbatim on an array
    pcd_points = np.stack([r.uniform(-2000, 2000, 700), r.uniform(-1500, 1200, 700), r.uniform(500, 4000, 700)], axis=1)
    pcd_points[:250, 1] = 1200 + r.normal(0, 3, 250)
    pcd_points = pcd_points.astype(np.float32).astype(np.float64)
    out["band_cloud"] = pcd_points
    idx_lower = np.argwhere(pcd_points[:, 1] >= pcd_points[:, 1].max() - 200)
    idx_upper = np.argwhere(pcd_points[:, 1] < pcd_points[:, 1].max() - 200)
    out["band_lower_idx"] = idx_lower.reshape(-1)
    out["band_upper_idx"] = idx_upper.reshape(-1)

    # ---- kalman_filter
    traj = np.cumsum(r.normal(size=(40, 3)), axis=0) * 10.0
    out["kalman_in"] = traj
    out["kalman_out"] = ref_filtering.kalman_filter(traj)
    out["kalman_out_params"] = ref_filtering.kalman_filter(traj, ri=5, qi=2, fi=0.9, hi=1)

    np.savez_compressed(OUT, **out)
    print("wrote", OUT, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
