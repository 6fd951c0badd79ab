"""Re-processing saved clouds: ``floor_removal.py``'s body (band 200 mm, RANSAC 30 mm x 2000 hypotheses of 30 points, SOR
50 / 0.30, no voxel step) over a few hundred fused WFOV-scene clouds, through ``remove_floor_batch`` (one cloud-input
frame-engine pipeline) and through the per-cloud ``remove_floor`` loop, in one process, alternated ``--rounds`` times.

The clouds: ``--frames`` rendered WFOV frames (3 sensors) fused by the depth engine in millimetres with the voxel
downsample and SOR of ``filter_outliers`` (what a recording saved), each repeated under small deterministic rigid
motions up to ``--clouds`` clouds.  The two paths must give identical clouds (both draw RANSAC hypotheses from the same
counter-based generator); the script fails otherwise.  ``remove_floor_batch`` builds its pipeline inside every call, and
that cost is in its time.  A profiled run of the cloud pipeline gives the ``cloud_load`` kernel's algorithmic bytes over
its device time.

Prints one JSON line with clouds/s of every run, their medians, the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kinectpy_b200 import _cabi, synth  # noqa: E402
from kinectpy_b200.floor_removal import remove_floor, remove_floor_batch  # noqa: E402
from kinectpy_b200.geometry import PointCloud  # noqa: E402
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig  # noqa: E402
from tools.bench_c5 import card  # noqa: E402

HBM_BPS = 7.7e12       # HGX B200 data sheet, one GPU


def saved_clouds(frames, n, voxel):
    depth, tab, T = synth.render_sequence(synth.WFOV, frames, 3)
    cfg = PipelineConfig(n_sensors=3, pixels=synth.WFOV.pixels, scale=1.0, voxel_size=voxel, sor_k=20, sor_ratio=2.0,
                         do_floor=False, do_icp=False, n_streams=4)
    pipe = FramePipeline(cfg, tab, synth.scale_extrinsics(T, 1.0))
    fused = [o.points for o in pipe.run(depth, want_points=True)]
    pipe.close()
    out = []
    for i in range(n):
        a = np.radians(0.5 * (i % 7) - 1.5)
        R = np.array([[np.cos(a), 0.0, np.sin(a)], [0.0, 1.0, 0.0], [-np.sin(a), 0.0, np.cos(a)]])
        t = np.array([3.0 * (i % 5) - 6.0, 0.0, 2.0 * (i % 3)])
        out.append(np.ascontiguousarray(fused[i % frames].astype(np.float64) @ R.T + t, np.float32))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8, help="rendered frames the clouds come from")
    ap.add_argument("--clouds", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--voxel", type=float, default=10.0, help="voxel of the fusion that made the saved clouds (mm)")
    ap.add_argument("--spacing", type=float, default=None, help="typical point spacing of the clouds (mm; default: --voxel)")
    ap.add_argument("--out", default=None, help="write the JSON line here as well")
    a = ap.parse_args()
    a.spacing = a.voxel if a.spacing is None else a.spacing
    clouds = saved_clouds(a.frames, a.clouds, a.voxel)
    pcds = [PointCloud(c) for c in clouds]

    # warm-up of both paths, and the identity check on every cloud
    batch = remove_floor_batch(pcds, spacing=a.spacing)
    loop = [remove_floor(p) for p in pcds]
    mismatch = [i for i, (b, l) in enumerate(zip(batch, loop)) if not np.array_equal(b.points, l.points)]
    if mismatch:
        raise SystemExit("remove_floor_batch and remove_floor differ on clouds %s" % mismatch[:10])

    runs = {"batch": [], "loop": []}
    ctx = _cabi.default_context()
    for _ in range(a.rounds):
        t0 = time.perf_counter()
        remove_floor_batch(pcds, spacing=a.spacing)
        runs["batch"].append(len(pcds) / (time.perf_counter() - t0))
        t0 = time.perf_counter()
        out = [remove_floor(p) for p in pcds]
        ctx.sync()
        runs["loop"].append(len(pcds) / (time.perf_counter() - t0))
        del out

    # the load kernel: algorithmic bytes over device time, in the engine's profiling mode
    cap = max(len(c) for c in clouds)
    cfg = PipelineConfig(input_mode=_cabi.INPUT_CLOUDS, cloud_voxel=0, n_sensors=1, pixels=cap, scale=1.0, voxel_size=a.spacing,
                         sor_k=0, floor_band=200.0, ransac_thr=30.0, ransac_n=30, ransac_iters=2000, floor_sor_k=50,
                         floor_sor_ratio=0.30, do_icp=False, n_streams=16)
    pipe = FramePipeline(cfg)
    pipe.profile(True)
    pipe.run_clouds(pcds)
    prof = pipe.profile_read()
    pipe.profile(False)
    pipe.close()
    load = prof.get("cloud_load", {"ms": float("nan"), "bytes": 0.0, "calls": 0})
    bps = load["bytes"] / (load["ms"] * 1e-3) if load["ms"] > 0 else float("nan")
    rec = {
        "card": card(),
        "voxel_mm": a.voxel, "spacing_mm": a.spacing, "clouds": len(clouds), "rows_mean": float(np.mean([len(c) for c in clouds])),
        "clouds_per_s": {k: [round(x, 2) for x in v] for k, v in runs.items()},
        "median_clouds_per_s": {k: round(statistics.median(v), 2) for k, v in runs.items()},
        "identical": True,
        "cloud_load": {"ms": load["ms"], "calls": load["calls"], "bytes": load["bytes"], "bytes_per_s": bps,
                       "share_of_7.7TB/s": bps / HBM_BPS},
        "profiled_families_ms": {k: round(v["ms"], 3) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])[:8]},
    }
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
