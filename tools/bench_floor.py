"""The frame engine's floor stage: what the reported plane costs in bench.py's configuration, and RANSAC mode against
plane mode at the reference's floor settings.

Two parts, both on one GPU in one process session:

1. ``--parent DIR`` (a built checkout of the commit before the plane was reported): ``bench.py --gpus 1 --steps S
   --warmup W --no-cpu-baseline --dump-outputs`` from DIR and from this tree, alternated ``--rounds`` times.  Every
   bench line is written under ``--out-dir`` and the dumps of each pair are compared byte for byte.
2. Reference floor settings (floor_removal.py:64-73: band 200 mm, RANSAC 30 mm x 2000 hypotheses of 30 points, SOR
   50 / 0.30) in millimetres on bench.py's shape (WFOV 3 x 1024^2, depth resident, 16 frames in flight), RANSAC mode
   against plane mode with the plane RANSAC mode reported for frame 0 (normal turned towards the floor, d moved by the
   threshold), alternated ``--rounds`` times; per-frame device time of the floor stage from the engine's profiling mode.

Prints one JSON line with the card's name and power limit read in the same run.
"""
import argparse
import filecmp
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kinectpy_b200 import _cabi, synth  # noqa: E402
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig  # noqa: E402
from tools.bench_c5 import card  # noqa: E402

FLOOR_FAMILIES = ("band_mask", "ransac_fit", "ransac_score", "ransac_select", "floor_refit", "plane_side", "floor_sor")


def same_tree(a, b):
    """Byte-identical directories (same file names, same contents)."""
    d = filecmp.dircmp(a, b)
    if d.left_only or d.right_only or d.funny_files:
        return False
    _, mismatch, errors = filecmp.cmpfiles(a, b, d.common_files, shallow=False)
    return not mismatch and not errors and all(same_tree(os.path.join(a, s), os.path.join(b, s)) for s in d.common_dirs)


def bench_pairs(a, tmp):
    runs = {"parent": [], "change": []}
    dumps_equal = []
    for r in range(a.rounds):
        dumps = {}
        for name, tree in (("parent", os.path.abspath(a.parent)), ("change", ROOT)):
            dump = os.path.join(tmp, "%s_%d" % (name, r))
            cmd = [sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", str(a.steps), "--warmup",
                   str(a.warmup), "--no-cpu-baseline", "--dump-outputs", dump]
            out = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, timeout=3600)
            if out.returncode != 0:
                sys.exit("bench_floor: bench.py failed in %s:\n%s" % (tree, out.stderr[-4000:]))
            line = json.loads([x for x in out.stdout.splitlines() if x.startswith("{")][-1])
            with open(os.path.join(a.out_dir, "r06_bench_%s_%d.json" % (name, r + 1)), "w") as f:
                f.write(json.dumps(line) + "\n")
            runs[name].append(line)
            dumps[name] = dump
        dumps_equal.append(same_tree(dumps["parent"], dumps["change"]))
    summary = {}
    for name, lines in runs.items():
        summary[name] = {"frames_per_s": [round(x["value"], 2) for x in lines], "gpu_launches": [x.get("gpu_launches") for x in lines],
                         "launches_per_frame": [x.get("launches_per_frame") for x in lines],
                         "e2e_d2h_bytes_per_step": [x["e2e"]["d2h_bytes_per_step"] for x in lines],
                         "e2e_frames_per_s": [round(x["e2e"]["value"], 2) for x in lines]}
    summary["dumps_identical"] = dumps_equal
    summary["frames_per_step"] = runs["change"][0]["config"]["frames_per_step_per_gpu"]
    return summary


def reference_floor(a):
    mode, S = synth.WFOV, 3
    depth, tab, T = synth.render_sequence(mode, 2, S)
    Tm = synth.scale_extrinsics(T, 1.0)
    Ti = np.stack([synth.perturbed_extrinsic(Tm[s], 0.3, (3, -3, 3), unit_scale=1.0) if s else Tm[s] for s in range(S)])
    mm = dict(n_sensors=S, pixels=mode.pixels, n_streams=a.streams, scale=1.0, voxel_size=10.0, floor_band=200.0,
              ransac_thr=30.0, ransac_n=30, ransac_iters=2000, floor_sor_k=50, floor_sor_ratio=0.30, icp_voxel=10.0,
              icp_max_corr=20.0, normals_radius=20.0)
    idx = np.arange(a.frames) % 2
    ran = FramePipeline(PipelineConfig(**mm), tab, Tm, Ti)
    buf_r = ran._ctx.to_device(depth[idx], np.uint16)
    ran._ctx.sync()
    first = ran.run(depth[:1])[0]
    plane = [float(x) for x in first.floor_plane]
    s = 1.0 if plane[1] > 0 else -1.0
    cut_plane = (s * plane[0], s * plane[1], s * plane[2], s * plane[3] + mm["ransac_thr"])
    cut = FramePipeline(PipelineConfig(**mm, floor_mode=_cabi.FLOOR_PLANE, floor_plane=cut_plane), tab, Tm, Ti)
    buf_c = cut._ctx.to_device(depth[idx], np.uint16)
    cut._ctx.sync()
    pipes = {"ransac": (ran, buf_r), "plane": (cut, buf_c)}

    def step(name):
        p, b = pipes[name]
        return p.run_raw(b.ptr, True, a.frames)

    fps = {k: [] for k in pipes}
    for name in pipes:
        for _ in range(a.warmup):
            step(name)
    for _ in range(a.rounds):
        for name in pipes:
            t0 = time.perf_counter()
            for _ in range(a.steps):
                step(name)
            fps[name].append(a.steps * a.frames / (time.perf_counter() - t0))
    res = {name: step(name) for name in pipes}
    counts = {name: {k: [int(getattr(res[name][f], k)) for f in range(2)] for k in ("n_sor", "n_floor_inliers", "n_out")}
              for name in pipes}
    prof, launches = {}, {}
    for name, (p, _) in pipes.items():
        l0 = p.launch_count()
        step(name)
        launches[name] = (p.launch_count() - l0) / a.frames
        p.profile(True)
        step(name)
        fam = p.profile_read()
        p.profile(False)
        prof[name] = {k: round(v["ms"] / a.frames, 5) for k, v in fam.items() if k in FLOOR_FAMILIES}
    for p, _ in pipes.values():
        p.close()
    med = {k: statistics.median(v) for k, v in fps.items()}
    return {"settings_mm": {k: mm[k] for k in ("voxel_size", "floor_band", "ransac_thr", "ransac_n", "ransac_iters", "floor_sor_k",
                                               "floor_sor_ratio")},
            "frames_per_call": a.frames, "streams": a.streams, "reported_plane_frame0": plane, "cut_plane": list(cut_plane),
            "frames_per_s": fps, "median_frames_per_s": med, "plane_over_ransac": med["plane"] / med["ransac"],
            "ms_per_frame_saved_end_to_end": 1e3 / med["ransac"] - 1e3 / med["plane"],
            "launches_per_frame": launches, "counts": counts, "profile_ms_per_frame": prof}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", default=None, help="built checkout of the parent commit (part 1; skipped without it)")
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frames", type=int, default=64, help="frames per timed call (part 2)")
    ap.add_argument("--streams", type=int, default=16)
    a = ap.parse_args()
    if not _cabi.device_available():
        sys.exit("bench_floor: no CUDA device (there is no CPU path to measure)")
    os.makedirs(a.out_dir, exist_ok=True)
    line = {"card": card()}
    with tempfile.TemporaryDirectory() as tmp:
        if a.parent:
            line["bench_parent_vs_change"] = bench_pairs(a, tmp)
    line["reference_floor_mm"] = reference_floor(a)
    s = json.dumps(line)
    print(s)
    with open(os.path.join(a.out_dir, "r06_bench_floor.json"), "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
