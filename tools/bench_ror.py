"""The frame engine's radius outlier removal (remove_radius_outlier after the SOR) at bench.py's shape.

One process, two configurations of the device-resident leg of bench.py (WFOV 3 x 1024^2, depth resident in HBM, 16
frames in flight), alternated --rounds times so that drift hits both alike:

    c4      the engine as bench.py runs it
    c4_ror  + the radius filter (nb_points --nb, radius --radius m)

The setting is our choice: the reference never calls remove_radius_outlier.  Prints one JSON line: frames/s of every
run and their medians, the card's name and power limit, the per-frame device time of the stage and of the SOR it
follows from the engine's profiling mode (one batch slot, direct launches), and for context the single-cloud
``kp_radius_mask`` (warp-per-query ring kernel, host round trip) on one frame's SOR output.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kinectpy_b200 import _cabi, synth  # noqa: E402
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig  # noqa: E402
from tools.bench_c5 import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64, help="frames per timed call")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--streams", type=int, default=16)
    ap.add_argument("--nb", type=int, default=8)
    ap.add_argument("--radius", type=float, default=0.03)
    ap.add_argument("--mask-reps", type=int, default=20, help="kp_radius_mask calls timed")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if not _cabi.device_available():
        sys.exit("bench_ror: no CUDA device (there is no CPU path to measure)")
    mode, S = synth.WFOV, 3
    depth, tab, T = synth.render_sequence(mode, 2, S)
    Ti = np.stack([synth.perturbed_extrinsic(T[s]) if s else T[s] for s in range(S)])
    idx = np.arange(a.frames) % 2
    configs = {
        "c4": PipelineConfig(n_sensors=S, pixels=mode.pixels, n_streams=a.streams),
        "c4_ror": PipelineConfig(n_sensors=S, pixels=mode.pixels, n_streams=a.streams, ror_nb_points=a.nb, ror_radius=a.radius),
    }
    pipes, bufs = {}, {}
    for name, cfg in configs.items():
        p = FramePipeline(cfg, tab, T, Ti)
        bufs[name] = p._ctx.to_device(depth[idx], np.uint16)
        p._ctx.sync()
        pipes[name] = p

    def step(name):
        return pipes[name].run_raw(bufs[name].ptr, True, a.frames)

    fps = {k: [] for k in configs}
    for name in configs:
        for _ in range(a.warmup):
            step(name)
    for _ in range(a.rounds):
        for name in configs:
            t0 = time.perf_counter()
            for _ in range(a.steps):
                step(name)          # (each call returns after its frames' records are on the host)
            fps[name].append(a.steps * a.frames / (time.perf_counter() - t0))
    res = {name: step(name) for name in configs}
    counts = {name: {"n_sor": [int(res[name][f].n_sor) for f in range(2)], "n_out": [int(res[name][f].n_out) for f in range(2)]}
              for name in configs}
    counts["c4_ror"]["n_ror"] = pipes["c4_ror"].frame_counts()["n_ror"]
    prof = {}
    for name in configs:
        p = pipes[name]
        p.profile(True)
        step(name)
        fam = p.profile_read()
        p.profile(False)
        prof[name] = {k: v["ms"] / a.frames for k, v in fam.items() if k in ("sor", "ror", "ror_count", "floor_sor")}
    # context: the single-cloud call on frame 0's SOR output (engine without floor removal: its final cloud)
    p = FramePipeline(PipelineConfig(n_sensors=S, pixels=mode.pixels, n_streams=1, do_floor=False, do_icp=False), tab, T, Ti)
    cloud = p.run(depth[:1], want_points=True)[0].points
    p.close()
    ctx = _cabi.default_context()
    d = ctx.to_device(np.ascontiguousarray(cloud, np.float32), np.float32)
    keep = ctx.empty((len(cloud),), np.uint8)
    kept = C.c_int64()
    for _ in range(2):
        ctx.check(ctx.lib.kp_radius_mask(ctx.handle, d.ptr, len(cloud), a.nb, a.radius, keep.ptr, None, C.byref(kept)))
    t0 = time.perf_counter()
    for _ in range(a.mask_reps):
        ctx.check(ctx.lib.kp_radius_mask(ctx.handle, d.ptr, len(cloud), a.nb, a.radius, keep.ptr, None, C.byref(kept)))
    ctx.sync()
    mask_ms = (time.perf_counter() - t0) * 1e3 / a.mask_reps
    base = statistics.median(fps["c4"])
    line = {"card": card(), "mode": "WFOV", "sensors": S, "frames_per_call": a.frames, "streams": a.streams, "steps": a.steps,
            "rounds": a.rounds, "ror_nb_points": a.nb, "ror_radius_m": a.radius,
            "frames_per_s": fps, "median_frames_per_s": {k: statistics.median(v) for k, v in fps.items()},
            "ratio_vs_c4": {k: statistics.median(v) / base for k, v in fps.items()}, "counts": counts,
            "profile_ms_per_frame": prof,
            "kp_radius_mask": {"points": int(len(cloud)), "kept": int(kept.value), "ms_per_call": mask_ms}}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")
    for p in pipes.values():
        p.close()


if __name__ == "__main__":
    main()
