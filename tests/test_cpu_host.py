"""CPU-side checks (no GPU needed): the C ABI library loads and exports every symbol the header
declares, the Python surface fails loudly without a device, host-side formats and the frame
sharding logic (world_size 2 over gloo)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "kp_api.h")).read()
    return sorted(set(re.findall(r"KP_EXPORT\s+[\w\s\*]+?\b(kp_\w+)\s*\(", txt)))


def test_header_symbols_are_exported_and_bound():
    from kinectpy_b200 import _cabi
    lib = _cabi.load_library()
    syms = header_symbols()
    assert len(syms) >= 40
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in kp_api.h but not exported by the library"
        assert s in _cabi.SIGNATURES, f"{s} has no ctypes prototype"
    assert sorted(_cabi.SIGNATURES) == syms
    assert b"sm_100a" in lib.kp_version()


def test_library_is_sm100a_only_and_has_tma():
    so = os.path.join(ROOT, "kinectpy_b200", "libkinectpy_b200.so")
    out = subprocess.run(["cuobjdump", "-lelf", so], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    assert "UBLKCP" in sass              # cp.async.bulk (TMA) staging of the calibration table in K1
    assert "SYNCS.ARRIVE.TRANS64" in sass  # mbarrier expect_tx that the bulk copy completes on


def test_no_cpu_fallback_without_device():
    from kinectpy_b200 import _cabi, PointCloud, KinectPyB200Error
    if _cabi.device_available():
        pytest.skip("a GPU is present")
    pcd = PointCloud(np.random.rand(100, 3))
    for call in (lambda: pcd.voxel_down_sample(0.1), lambda: pcd.remove_statistical_outlier(5, 1.0),
                 lambda: pcd.segment_plane(0.01, 3, 10), lambda: pcd.estimate_normals()):
        with pytest.raises(KinectPyB200Error):
            call()
    # host-only attribute handling still works (it is not compute)
    assert len(pcd) == 100 and np.asarray(pcd.points).shape == (100, 3)


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "kinectpy_b200")):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, fn)).read()
                assert "oracle" not in txt.lower() or fn in ("kp_ransac.cu", "kp_grid.cu", "kp_primitives.cu", "kp_common.cuh"), fn
                assert "import oracle" not in txt and "from oracle" not in txt and "kp_oracle" not in txt, fn


def test_pcd_roundtrip_host_only(tmp_path):
    from kinectpy_b200 import PointCloud
    from kinectpy_b200.io_formats import read_point_cloud, write_point_cloud
    r = np.random.default_rng(0)
    pcd = PointCloud(r.normal(size=(257, 3)) * 1000)
    pcd.colors = r.integers(0, 256, (257, 3)) / 255.0
    for ascii_ in (False, True):
        fp = str(tmp_path / f"c{int(ascii_)}.pcd")
        write_point_cloud(fp, pcd, write_ascii=ascii_)
        back = read_point_cloud(fp)
        assert np.array_equal(np.asarray(back.points, np.float32), np.asarray(pcd.points, np.float32))
        assert np.allclose(back.colors, pcd.colors, atol=1e-9)
    empty = str(tmp_path / "e.pcd")
    write_point_cloud(empty, PointCloud())
    assert len(read_point_cloud(empty)) == 0


def test_depth_dat_layout(tmp_path):
    from kinectpy_b200.utils import io as kio
    a = np.arange(-30, 30, dtype=np.int16).reshape(-1, 3)
    kio.save_depth(str(tmp_path / "17"), a)
    assert os.path.exists(tmp_path / "17_depth.dat")
    assert np.array_equal(kio.load_depth(str(tmp_path / "17")), a)
    assert np.array_equal(kio.load_depth(str(tmp_path / "17_depth.dat")), a)


def test_reference_surface_signatures():
    import inspect
    from kinectpy_b200.preprocessing import filtering, registration
    from kinectpy_b200 import floor_removal
    from kinectpy_b200.utils import io as kio
    sig = lambda f: [(p.name, p.default) for p in inspect.signature(f).parameters.values()]
    E = inspect.Parameter.empty
    assert sig(filtering.filter_outliers) == [("pcd", E), ("nb_neighbors", 200), ("std_ratio", 3.0), ("voxel_size", 0.02)]
    assert sig(filtering.kalman_filter) == [("joint_vals", E), ("ri", 10), ("qi", 10), ("fi", 1 / 30), ("hi", 1)]
    assert sig(registration.preprocess_point_cloud) == [("pcd", E), ("voxel_size", E), ("normals_nn", 30), ("fpfh_nn", 100)]
    assert sig(registration.prepare_dataset) == [("pcd_master", E), ("pcd_sub", E), ("voxel_size", E), ("normals_nn", 40), ("fpfh_nn", 40)]
    assert sig(registration.execute_global_registration) == [("pcd_master", E), ("pcd_sub", E), ("voxel_size", 35), ("ransac_n_trials", 15)]
    assert sig(registration.execute_point_to_plane_registration)[:4] == [("pcd_master", E), ("pcd_sub", E), ("initial_transformation", E), ("voxel_size", 35)]
    assert sig(registration.execute_colored_ICP_registration)[:3] == [("pcd_master", E), ("pcd_sub", E), ("initial_transformation", E)]
    assert sig(floor_removal.equation_plane) == [("p1", E), ("p2", E), ("p3", E)]
    assert sig(floor_removal.pcd_above_plane) == [("a", E), ("b", E), ("c", E), ("d", E), ("pcd", E)]
    assert sig(kio.rgbd_to_pointcloud)[:2] == [("color_img", E), ("depth_img", E)]
    assert floor_removal.equation_plane((0, 0, 0), (1, 0, 0), (0, 1, 0)) == (0, 0, 1, 0)


def test_kalman_filter_restatement():
    from kinectpy_b200.preprocessing.filtering import kalman_filter
    z = np.cumsum(np.random.default_rng(1).normal(size=(50, 3)), 0)
    x = kalman_filter(z)
    assert x.shape == z.shape and np.array_equal(x[0], z[0]) and np.isfinite(x).all()


def test_synthetic_scene_statistics():
    from kinectpy_b200 import synth
    for mode, frac in ((synth.NFOV, 0.75), (synth.WFOV, 0.785)):
        tab = synth.xy_table(mode)
        assert tab.shape == (mode.pixels, 2) and abs((~np.isnan(tab[:, 0])).mean() - frac) < 0.01
    T = synth.extrinsics(3)
    assert np.allclose(T[0], np.eye(4)) and np.allclose(np.linalg.det(T[:, :3, :3]), 1)
    d0 = synth.render_depth(synth.NFOV, T[1], 3, 1)
    d1 = synth.render_depth(synth.NFOV, T[1], 3, 1)
    assert np.array_equal(d0, d1) and d0.dtype == np.uint16 and 0.70 < (d0 > 0).mean() < 0.75


def test_frame_sharding_partition():
    from kinectpy_b200.sharding import frames_for_rank
    for F in (0, 1, 7, 1000):
        for G in (1, 2, 4, 8):
            parts = [frames_for_rank(F, r, G) for r in range(G)]
            allf = np.sort(np.concatenate(parts)) if F else np.zeros(0, np.int64)
            assert np.array_equal(allf, np.arange(F)) and max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


_WORKER = r'''
import os, sys
import numpy as np
import torch.distributed as dist
sys.path.insert(0, os.environ["KP_ROOT"])
from kinectpy_b200.sharding import frames_for_rank, gather_frame_results
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["KP_PORT"],
                        rank=int(os.environ["RANK"]), world_size=2)
rank, F = dist.get_rank(), 7
mine = frames_for_rank(F, rank, 2)
T = np.stack([np.stack([np.eye(4) * (f + 1), np.eye(4) * -(f + 1)]) for f in mine])
counts = np.stack([[f * 10, f * 10 + 1, f * 10 + 2] for f in mine]).astype(np.int64)
allT, allc = gather_frame_results(mine, T, counts, F)
assert allT.shape == (F, 2, 4, 4) and all(allT[f, 0, 0, 0] == f + 1 and allT[f, 1, 1, 1] == -(f + 1) for f in range(F))
assert np.array_equal(allc[:, 0], np.arange(F) * 10)
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
'''


def test_gather_epilogue_world_size_2_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), KP_ROOT=ROOT, KP_PORT=port)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs


def test_bench_reference_arm_line_contract():
    """`bench.py --impl reference` (the CPU arm the driver times next to ours) prints ONE JSON line with the contract's
    keys, runs on every host thread even when a launcher exported OMP_NUM_THREADS=1 (torchrun does), and needs no GPU."""
    import json
    import subprocess
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--mode", "NFOV", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "fused_3kinect_frames_per_s" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_bench_b200_arm_fails_loudly_without_a_gpu():
    """No silent CPU fallback in the measured arm either: without a CUDA device `bench.py` exits non-zero and says why
    (the CPU arm is a separate, explicitly requested `--impl reference`)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout) and not any(ln.startswith("{") for ln in r.stdout.splitlines())


def test_bench_dump_outputs_arrays():
    """`bench.py --dump-outputs`: every field of the per-frame results as float64, and the final clouds as float32 -- all
    valid rows when they fit, else the same seeded sample of (frame, row) pairs on every run -- within 64 MB."""
    sys.path.insert(0, ROOT)
    import bench
    from kinectpy_b200 import _cabi
    res = (_cabi.FrameResult * 2)()
    res[1].n_out, res[1].icp_T[0][3], res[1].icp_iters[1] = 5, 0.25, 7
    a = bench.result_arrays(res, 3)
    assert a["icp_T"].shape == (2, 2, 4, 4) and a["icp_T"][1, 0, 0, 3] == 0.25 and a["icp_iters"][1, 1] == 7
    assert a["n_out"].tolist() == [0, 5] and all(v.dtype == np.float64 for v in a.values())
    xyz = np.random.default_rng(0).normal(size=(3, 10, 3)).astype(np.float32)
    full = bench.cloud_sample(xyz, [4, 0, 10])
    assert np.array_equal(full["points"], np.concatenate([xyz[0, :4], xyz[2]])) and full["points_index"].dtype == np.float32
    s = bench.cloud_sample(xyz, [4, 0, 10], rows=6)
    f, r = s["points_index"].astype(np.int64).T
    assert len(f) == 6 and (r < np.array([4, 0, 10])[f]).all() and (np.diff(f * 10 + r) > 0).all()
    assert np.array_equal(s["points"], xyz[f, r]) and np.array_equal(s["points"], bench.cloud_sample(xyz, [4, 0, 10], rows=6)["points"])
    assert bench.DUMP_ROWS * (12 + 8) < 64e6
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + bad, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error" in r.stderr


def test_bench_gives_every_rank_the_same_workload():
    """Weak scaling needs the same per-GPU work on every rank: `bench.make_inputs` hands every rank the same distinct frames,
    rotated by rank (a first version gave rank r its own window of the synthetic sequence; the windows differed by up to
    11 % in cost and read as 0.91 scaling efficiency: profiles/r02_g_gpu_variance.json)."""
    sys.path.insert(0, ROOT)
    import bench
    base = bench.make_inputs("NFOV", 3, 0)
    for rank in (1, 2, 5):
        other = bench.make_inputs("NFOV", 3, rank)
        assert np.array_equal(np.roll(base[1], -(rank % 3), axis=0), other[1])       # same frames, rotated
        for a, b in zip(base[2:], other[2:]):
            assert np.array_equal(a, b, equal_nan=True)                               # same tables and extrinsics
