"""BASELINE config C5 on the frame engine: the human crop and the fixed-N PointNet batch from the same call.

One process, three configurations of the device-resident leg of bench.py (WFOV 3 x 1024^2, depth and segmentation
images resident in HBM, 16 frames in flight), alternated --rounds times so that drift hits each of them alike:

    c4            the engine as bench.py runs it
    c4_crop       + the human crop (crop_gate --gate mm)
    c4_crop_fixed + the crop + a [F, N, 3] fixed-N RANDOM output (N = --n)

Prints one JSON line: frames/s of every run, their medians, the card's name and power limit, and the per-family
device times of the crop and resample kernels from the engine's profiling mode (one batch slot, direct launches).
How much the crop speeds up the later stages is measured here only as the difference of the frame rates.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kinectpy_b200 import _cabi, synth  # noqa: E402
from kinectpy_b200.pipeline import FramePipeline, PipelineConfig  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:      # (reported, not fatal: the numbers are still the run's)
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64, help="frames per timed call")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--streams", type=int, default=16)
    ap.add_argument("--gate", type=float, default=1500.0)
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if not _cabi.device_available():
        sys.exit("bench_c5: no CUDA device (there is no CPU path to measure)")
    mode, S = synth.WFOV, 3
    depth, tab, T = synth.render_sequence(mode, 2, S)
    rgb = np.stack([np.stack([synth.render_segmentation(mode, T[s], f, s, table=tab[s]) for s in range(S)]) for f in range(2)])
    Ti = np.stack([synth.perturbed_extrinsic(T[s]) if s else T[s] for s in range(S)])
    idx = np.arange(a.frames) % 2
    configs = {
        "c4": PipelineConfig(n_sensors=S, pixels=mode.pixels, n_streams=a.streams),
        "c4_crop": PipelineConfig(n_sensors=S, pixels=mode.pixels, n_streams=a.streams, do_crop=True, crop_gate=a.gate),
        "c4_crop_fixed": PipelineConfig(n_sensors=S, pixels=mode.pixels, n_streams=a.streams, do_crop=True, crop_gate=a.gate,
                                        resample_n=a.n, resample_mode=_cabi.RESAMPLE_RANDOM),
    }
    pipes, bufs = {}, {}
    for name, cfg in configs.items():
        p = FramePipeline(cfg, tab, T, Ti)
        d = p._ctx.to_device(depth[idx], np.uint16)
        r = p._ctx.to_device(rgb[idx], np.uint8) if cfg.do_crop else None
        fx = p._ctx.empty((a.frames, a.n, 3), np.float32) if cfg.resample_n else None
        p._ctx.sync()
        pipes[name], bufs[name] = p, (d, r, fx)

    def step(name):
        p = pipes[name]
        d, r, fx = bufs[name]
        res = (_cabi.FrameResult * a.frames)()
        rc = p.lib.kp_pipeline_run_ex(p.handle, d.ptr, r.ptr if r is not None else None, 1, a.frames, None, res, None, 0,
                                      fx.ptr if fx is not None else None)
        if rc != 0:
            p._raise(rc)
        return res

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
    res = step("c4_crop_fixed")
    n_out = [int(res[f].n_out) for f in range(2)]
    prof = {}
    for name in ("c4_crop", "c4_crop_fixed"):
        p = pipes[name]
        p.profile(True)
        step(name)
        fam = p.profile_read()
        p.profile(False)
        prof[name] = {k: v for k, v in fam.items() if k.startswith(("crop", "unproject", "resample"))}
        prof[name]["per_frame_ms"] = {k: v["ms"] / a.frames for k, v in fam.items() if k.startswith(("crop", "unproject", "resample"))}
    base = statistics.median(fps["c4"])
    line = {"card": card(), "mode": "WFOV", "sensors": S, "frames_per_call": a.frames, "streams": a.streams, "steps": a.steps,
            "rounds": a.rounds, "crop_gate_mm": a.gate, "resample_n": a.n,
            "frames_per_s": fps, "median_frames_per_s": {k: statistics.median(v) for k, v in fps.items()},
            "speedup_vs_c4": {k: statistics.median(v) / base for k, v in fps.items()},
            "final_points_with_crop": n_out, "profile": prof}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")
    for p in pipes.values():
        p.close()


if __name__ == "__main__":
    main()
