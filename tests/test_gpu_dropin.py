"""Drop-in test on the reference's OWN source text.

The reference's hot-path wrappers -- ``filter_outliers`` (preprocessing/filtering.py:12-25),
``preprocess_point_cloud`` / ``prepare_dataset`` / ``execute_point_to_plane_registration``
(preprocessing/registration.py:7-29, 65-86), the loop body of floor_removal.py (:63-73) and the fusion body of
``DataProcessor``'s frame loop (preprocessing/data.py:41-61) -- are executed UNMODIFIED with ``o3d`` bound to
``kinectpy_b200.o3d`` (the import swap of INTEGRATION.md) on the B200, and their results are compared with
tests/golden/reference_compositions.npz, which the same source produced over the CPU oracle
(tests/golden/make_composition_golden.py).  The source text is the fixture's: the generator stored it verbatim."""
import contextlib
import copy
import io
import os
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(HERE, "golden", "reference_compositions.npz"))


def shim():
    import kinectpy_b200.o3d as o3d
    return o3d


def cloud(o3d, pts, colors=None):
    pcd = o3d.geometry.PointCloud()
    pcd.points = o3d.utility.Vector3dVector(np.asarray(pts, np.float64))
    if colors is not None:
        pcd.colors = o3d.utility.Vector3dVector(np.asarray(colors, np.float64))
    return pcd


def reference_functions(gold, names, key):
    """The reference's functions, compiled from its own source with `o3d` = the B200 shim."""
    ns = {"o3d": shim(), "np": np, "copy": copy}
    exec(str(gold[key]), ns)
    assert all(n in ns for n in names)
    return ns


def test_reference_filter_outliers_runs_on_the_gpu_library(gold):
    o3d = shim()
    fn = reference_functions(gold, ["filter_outliers"], "fo_source")["filter_outliers"]
    src = cloud(o3d, gold["fo_in"])
    out = fn(src, nb_neighbors=20, std_ratio=2.0, voxel_size=0.02)
    assert np.array_equal(np.asarray(out.points, np.float32), gold["fo_out"])
    assert np.array_equal(np.asarray(src.points, np.float32), gold["fo_in"])          # input untouched (deepcopy at filtering.py:23)
    # the reference's defaults on millimetre data (200 neighbours, every point its own voxel)
    out = fn(cloud(o3d, gold["fo_default_in"]))
    assert np.array_equal(np.asarray(out.points, np.float32), gold["fo_default_out"])


def test_reference_point_to_plane_registration_runs_on_the_gpu_library(gold):
    o3d = shim()
    ns = reference_functions(gold, ["preprocess_point_cloud", "prepare_dataset", "execute_point_to_plane_registration"], "reg_source")
    with contextlib.redirect_stdout(io.StringIO()):
        T = ns["execute_point_to_plane_registration"](cloud(o3d, gold["reg_master"]), cloud(o3d, gold["reg_sub"]), gold["reg_init"], voxel_size=35)
    T = np.asarray(T, np.float64)
    assert np.abs(T[:3, :3] - gold["reg_T"][:3, :3]).max() < 1e-4
    assert np.abs(T[:3, 3] - gold["reg_T"][:3, 3]).max() < 1e-4 * 1000.0       # millimetre units


def test_reference_floor_removal_body_runs_on_the_gpu_library(gold):
    o3d = shim()
    o3d.utility.random.seed(1234)
    ns = {"np": np, "o3d": o3d, "pcd": cloud(o3d, gold["floor_in"])}
    exec(str(gold["floor_source"]), ns)
    assert np.array_equal(np.asarray(ns["inliers"], np.int64), gold["floor_inliers"])
    assert np.allclose(np.asarray(ns["plane_model"], np.float64), gold["floor_plane"], rtol=0, atol=1e-9 * 1000)
    assert np.array_equal(np.asarray(ns["filtered_pcd"].points, np.float32), gold["floor_out"])


def test_reference_fusion_body_runs_on_the_gpu_library(gold):
    o3d = shim()
    fo = reference_functions(gold, ["filter_outliers"], "fo_source")["filter_outliers"]
    pcs = [cloud(o3d, c, np.full((len(c), 3), 0.5)) for c in gold["fuse_in"]]
    ns = {"np": np, "o3d": o3d, "filter_outliers": fo, "filtered_pcds": pcs,
          "self": types.SimpleNamespace(registration_transformations=[t for t in gold["fuse_T"]])}
    exec(str(gold["fuse_source"]), ns)
    assert np.array_equal(np.asarray(ns["registered_pcd"].points, np.float32), gold["fuse_out"])
