#!/usr/bin/env python
"""bench.py -- fused 3-Kinect frames/s of the B200 per-frame point-cloud path.

Workload (BASELINE.json configs[3], "C4"): a synthetic 3-sensor WFOV 1024x1024 depth sequence;
per frame unproject -> transform -> fuse -> 1 cm voxel -> SOR(20, 2.0) -> floor removal
(20 cm band, RANSAC 1 cm / 1000 hypotheses, merge, SOR(50, 0.30)) -> point-to-plane ICP refinement
of both sub extrinsics (1 cm voxel, normals r = 2 cm / 30 nn, max_corr 2 cm, <= 30 iterations).
A "step" is one call of the frame engine over --frames-per-step frames per rank; frames are sharded over
ranks with no collective on the frame path (weak scaling: per-GPU work is fixed).  The engine is driven by
ONE host thread per GPU: B frames per kernel launch, W batch slots in flight, one CUDA graph per slot.

  python bench.py --gpus 1 --steps K --warmup W            # our arm
  python bench.py --impl reference ...                     # CPU arm: the oracle port on the host cores
  torchrun ... bench.py --gpus N ...                       # one rank per GPU

Prints ONE JSON line on rank 0.  Beside the headline (C4) it carries driver-run legs for the other BASELINE
configs: C1 (1 x NFOV: voxel + SOR), C2 (3 x NFOV: ICP ms/pair), C3 (RANSAC on the fused WFOV cloud), C5 (resample).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fused_3kinect_frames_per_s"
UNIT = "frames/s"
ICP_START = {"angle_deg": 0.3, "shift_mm": [3, -3, 3]}     # ground truth perturbed by this much (see DESIGN.md 7)
SENSOR_YAW_DEG = [0.0, 40.0, -40.0]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="WFOV", choices=["WFOV", "NFOV"])
    ap.add_argument("--frames-per-step", type=int, default=0, help="frames per step and GPU (0 = 2 x frames in flight)")
    ap.add_argument("--distinct-frames", type=int, default=4, help="synthetic frames rendered per rank (cycled)")
    ap.add_argument("--streams", type=int, default=16, help="frames in flight per GPU (B frames per launch x W batch slots)")
    ap.add_argument("--cpu-sample-frames", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-resample", action="store_true", help="skip the config-C5 resampling leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-legs", action="store_true", help="skip the C1 / C2 / C3 legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (rank 0): the "
                         "per-frame results of the device-resident step and a seeded sample of the clouds of the e2e step")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons of THIS rank's GPU, sampled every 200 ms during the timed region through NVML
    inside the process (a thread that sleeps between two cheap queries).  Round 1 started one `nvidia-smi -lms`
    process per rank: eight of them disturbed the 8-GPU run they were meant to watch."""

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.sm, self.mx, self.reasons = [], [], set()
        self.stop_flag = threading.Event()
        self.th = None
        self.err = None

    def _loop(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.idx
            if vis:
                try:
                    idx = int(vis.split(",")[self.idx])
                except Exception:
                    pass
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            while not self.stop_flag.is_set():
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.mx.append(float(mx))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for name, b in bits.items():
                        if r & b:
                            self.reasons.add(name)
                except Exception:
                    pass
                self.stop_flag.wait(0.2)
        except Exception as e:       # no NVML: one nvidia-smi query instead of a loop
            self.err = repr(e)

    def start(self):
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag.set()
        if self.th:
            self.th.join(timeout=2)
        if not self.sm:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=10).stdout.strip().split(",")
                return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "reasons": [], "samples": 1, "source": "nvidia-smi after the region (NVML unavailable: %s)" % self.err}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": max(self.mx), "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "NVML, this rank's GPU, 200 ms period"}


def make_inputs(mode_name, distinct, rank, scale=1e-3, sensors=3):
    from kinectpy_b200 import synth
    mode = synth.MODES[mode_name]
    # Weak scaling: the per-GPU work is the same on every rank -- the same `distinct` frames, their order rotated by rank
    # (what round-robin sharding of a long recording gives every rank statistically).  Round 2 first gave rank r the
    # window [r * distinct, (r + 1) * distinct) of the synthetic sequence: those windows differ by up to 11 % in cost
    # (the figure moves through the room), which read as 0.91 scaling efficiency at 4 and 8 GPUs although every GPU,
    # alone on its window-0 data, ran the same 176 ms (profiles/r02_g_gpu_variance.json).
    depth, tab, T = synth.render_sequence(mode, distinct, sensors, first_frame=0)
    depth = np.roll(depth, -(rank % max(distinct, 1)), axis=0)
    T_fuse = synth.scale_extrinsics(T, scale)
    T_icp = np.stack([synth.perturbed_extrinsic(T_fuse[s], ICP_START["angle_deg"], tuple(ICP_START["shift_mm"]), unit_scale=scale) if s else T_fuse[s]
                      for s in range(sensors)])
    return mode, depth, tab, T_fuse, T_icp


def cpu_baseline(cfg, depth, tab, T_fuse, T_icp, frames):
    """The oracle port (oracle/kp_oracle.c, OpenMP over all host cores) on a bounded sample of the workload."""
    from oracle import oracle as orc
    orc.build()
    # every host thread this process may use, whatever OMP_NUM_THREADS a launcher exported
    orc.set_num_threads(int(os.environ.get("KP_REF_THREADS", len(os.sched_getaffinity(0)))))
    t0 = time.perf_counter()
    tm = {}
    for f in range(frames):
        orc.frame_pipeline(cfg, depth[f % depth.shape[0]], tab, T_fuse, T_icp, timings=tm)
    dt = time.perf_counter() - t0
    return {"value": frames / dt, "unit": UNIT, "cores": orc.num_threads(), "kind": "port",
            "sample": "%d frame(s) of the same workload, all stages, oracle/kp_oracle.c with OpenMP" % frames,
            "seconds": round(dt, 3), "stage_seconds": {k: round(v, 3) for k, v in tm.items()}}


# kernel family of the profile -> (dominant kernel, binding resource)
LEAF = {
    "knn_level0": ("k_knn_hist_b", "issue"), "knn_level1": ("k_knn_wbf_b", "issue"), "knn_stragglers": ("k_knn_b", "issue"),
    "knn_vbi": ("k_knn_vbi_b", "issue"), "knn_mid": ("k_knn_mid_b", "issue"), "icp": ("k_icp_iter_b", "issue"),
    "radix_sort": ("k_rs_scatter", "hbm"), "ransac_score": ("k_e_ransac_score", "fp64"), "ransac_fit": ("k_e_ransac_fit", "latency"),
    "ransac_select": ("k_e_ransac_select", "latency"),
    "unproject_transform": ("k_unproject", "hbm"), "voxel_mean": ("k_e_voxel_mean", "hbm"), "voxel_keys": ("k_e_voxel_keys", "hbm"),
    "grid_build": ("k_eg_scatter", "hbm"), "vbi_build": ("k_vbi_scatter", "hbm"), "compact_rows": ("k_bc_scatter", "hbm"),
    "compact_index": ("k_bc_scatter", "hbm"), "run_heads": ("k_bc_scatter", "hbm"), "sor_stats": ("k_bcsum_level", "hbm"),
    "band_mask": ("k_e_band_mask", "hbm"), "merge": ("k_e_append_rows", "hbm"),
}


def family_bytes(st, cfg, S, P, icp_iters=()):
    """Algorithmic HBM bytes per FRAME of every streaming family, from the frame's own counts (DESIGN.md 4).
    N = fused rows, Nv = valid, M = voxels, K = kept by SOR, lo = band, E = merged, per ICP cloud P rows."""
    NP = S * P
    Nv, M, K, E = st["n_fused"], st["n_voxel"], st["n_sor"], st["n_merged"]
    lo = st["n_lo"]
    icp = 1 if (cfg.do_icp and S > 1) else 0
    Mi = st["n_icp"]                                         # voxel counts of the S ICP clouds
    b = {}
    b["unproject_transform"] = NP * (2 + 12 + 12 * icp) + NP * 8
    b["voxel_keys"] = (NP + icp * NP) * (12 + 4)
    b["radix_sort"] = (NP + icp * NP) * (4 * 2 * 8 + 4)      # 4 passes x (key + index) read and written, one histogram read each
    b["run_heads"] = (Nv + icp * sum(st["nv_icp"])) * 2 * 4
    b["voxel_mean"] = (Nv + icp * sum(st["nv_icp"])) * (4 + 12) + (M + icp * sum(Mi)) * (12 + 4)
    # neighbour grids: level 0 + level 1 of SOR and floor SOR, level 0 + 1 of the ICP target: 12 B read per pass (4 passes) + rank / loc + 16 B row
    gpts = 2 * M + 2 * E + icp * 2 * Mi[0]
    b["grid_build"] = gpts * (3 * 12 + 4 * 4 + 16)
    b["sor_stats"] = (M + E) * (3 * 8 + 1)
    b["compact_rows"] = (M + K + lo + E) * (2 * 1 + 12) + (K + K + (lo - st["n_inl"]) + st["n_out"]) * 12
    b["compact_index"] = 2 * (2 * M + 2 * E + icp * 2 * Mi[0]) * 1
    b["band_mask"] = K * (2 * 12 + 1)
    b["merge"] = (K - lo) * 24
    b["ransac_score"] = lo * 12 + cfg.ransac_iters * 40
    b["knn_level0"] = (M + E + icp * Mi[0]) * 16 + (M + E) * 8 + icp * Mi[0] * 12
    # level-0 leftovers of the two SOR searches through the mid level: the query row + its output
    b["knn_mid"] = sum(st["leftovers_l0"][:2]) * (16 + 8)
    # a pass reads and rewrites the moving source (2 x 24 B) and its partner index (2 x 4 B), and gathers the partner's
    # row (16 B) and normal (12 B); pair i runs icp_iters[i] + 1 working passes over the points of sub cloud i + 1
    b["icp"] = float(sum((int(it) + 1) * 84 * Mi[i + 1] for i, it in enumerate(icp_iters))) if icp else 0.0
    return b


DUMP_ROWS = 1 << 21      # cloud rows --dump-outputs writes at most: 2 Mi rows x (12 + 8) B = 40 MiB of the 64 MB allowed


def result_arrays(res, S):
    """The kp_frame_result array a pipeline call returns, field by field, as float64 arrays (frame first)."""
    out = {k: np.array([getattr(r, k) for r in res], np.float64)
           for k in ("n_fused", "n_voxel", "n_sor", "n_floor_inliers", "n_out", "status")}
    out["icp_T"] = np.array([[list(r.icp_T[i]) for i in range(S - 1)] for r in res], np.float64).reshape(len(res), S - 1, 4, 4)
    for k in ("icp_fitness", "icp_rmse", "icp_iters"):
        out[k] = np.array([list(getattr(r, k))[:S - 1] for r in res], np.float64)
    return out


def cloud_sample(xyz, n_out, rows=DUMP_ROWS, seed=0):
    """Final clouds xyz float32 [F, stride, 3], of which the first n_out[f] rows of frame f are valid: all valid rows when
    there are at most `rows` of them, else a seeded uniform sample of `rows`, in (frame, row) order, with their indices."""
    off = np.concatenate([[0], np.cumsum(np.asarray(n_out, np.int64))])
    g = np.arange(off[-1]) if off[-1] <= rows else np.sort(np.random.default_rng(seed).choice(off[-1], rows, replace=False))
    f = np.searchsorted(off, g, side="right") - 1
    r = g - off[f]
    return {"points": np.ascontiguousarray(xyz[f, r], np.float32), "points_index": np.stack([f, r], 1).astype(np.float32)}


def write_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_pipeline_leg(ctx, cfg, depth, tab, T_fuse, T_icp, device, frames, steps):
    """frames/s of a pipeline configuration with depth resident in HBM (CUDA events on the ctx stream, L2 flushed)."""
    from kinectpy_b200.pipeline import FramePipeline
    pipe = FramePipeline(cfg, tab, T_fuse, T_icp, device=device)
    batch = np.ascontiguousarray(depth[np.arange(frames) % depth.shape[0]])
    d = pipe.upload(batch)
    for _ in range(3):
        res = pipe.run_raw(d.ptr, True, frames)
    ms = 0.0
    for _ in range(steps):
        ctx.flush_l2(); ctx.sync(); ctx.timer_start()
        res = pipe.run_raw(d.ptr, True, frames)
        ms += ctx.timer_stop()
    return pipe, d, res, ms / steps


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    from kinectpy_b200.pipeline import PipelineConfig
    mode_px = {"WFOV": 1024 * 1024, "NFOV": 640 * 576}[args.mode]
    cfg = PipelineConfig(n_sensors=3, pixels=mode_px, n_streams=args.streams)
    if args.frames_per_step <= 0:
        args.frames_per_step = 2 * args.streams
    workload = ("C4: 3 x %s synthetic depth frames -> unproject+transform+fuse -> voxel 1cm -> SOR(20,2.0) -> "
                "floor removal (band 20cm, RANSAC 1cm x1000, SOR(50,0.30)) -> p2plane ICP x2 (max_corr 2cm, <=30 it)" % args.mode)
    config = {"workload": workload, "mode": args.mode, "sensors": 3, "frames_per_step_per_gpu": args.frames_per_step,
              "distinct_frames": args.distinct_frames, "frames_in_flight_per_gpu": args.streams, "host_threads_per_gpu": 1,
              "host_cores": cores, "sharding": "frames are independent units, no collective; every rank runs the same distinct frames (order rotated by rank): per-GPU work fixed",
              "icp_start": "ground-truth extrinsic perturbed by %.1f deg about (1,1,1)/sqrt(3) and (%+d,%+d,%+d) mm" %
                           (ICP_START["angle_deg"], *ICP_START["shift_mm"]),
              "sensor_yaw_deg": SENSOR_YAW_DEG,
              "l2": "flushed between timed steps (256 MiB memset on the timing stream)",
              "arithmetic": "decisions and sums in f64 on f32-stored points (no FMA contraction); fp32 only pre-selects candidates"}

    # ------------------------------------------------------------------ reference arm (CPU oracle port)
    if args.impl == "reference":
        if rank != 0:
            return
        # torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm runs alone on rank 0 and is meant to use every
        # host thread it can get (KP_REF_THREADS overrides).  Set before the OpenMP runtime of the oracle library loads.
        os.environ["OMP_NUM_THREADS"] = os.environ.get("KP_REF_THREADS", str(cores))
        _, depth, tab, T_fuse, T_icp = make_inputs(args.mode, min(args.distinct_frames, 2), 0)
        from oracle import oracle as orc
        orc.build()
        orc.set_num_threads(int(os.environ["OMP_NUM_THREADS"]))
        for _ in range(min(args.warmup, 1)):
            orc.frame_pipeline(cfg, depth[0], tab, T_fuse, T_icp)
        t0 = time.perf_counter()
        for s in range(args.steps):
            orc.frame_pipeline(cfg, depth[s % depth.shape[0]], tab, T_fuse, T_icp)
        dt = time.perf_counter() - t0
        val = args.steps / dt
        cb = {"value": val, "unit": UNIT, "cores": orc.num_threads(), "kind": "port",
              "sample": "each step = 1 frame of the workload (bounded sample), oracle/kp_oracle.c with OpenMP on all host threads"}
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                          "data": "synthetic", "config": config, "cpu_baseline": cb,
                          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from kinectpy_b200 import _cabi
    from kinectpy_b200.pipeline import FramePipeline

    mode, depth, tab, T_fuse, T_icp = make_inputs(args.mode, args.distinct_frames, rank)
    S, P, B = 3, mode.pixels, args.frames_per_step
    pipe = FramePipeline(cfg, tab, T_fuse, T_icp, device=local_rank)
    fpl, slots = pipe.frames_in_flight()
    config["frames_per_launch"] = fpl
    config["batch_slots"] = slots
    ctx = _cabi.default_context(local_rank)
    batch = np.ascontiguousarray(depth[np.arange(B) % depth.shape[0]])      # uint16 [B,S,P]
    d_batch = pipe.upload(batch)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps, each bracketed by CUDA events on the ctx stream (a step call returns only after every batch
        slot's streams are drained, so the event pair spans the whole step); L2 flushed between steps.  Returns the
        summed time and what the last step returned."""
        total_ms, out = 0.0, None
        for _ in range(steps):
            ctx.flush_l2()
            ctx.sync()
            ctx.timer_start()
            out = fn()
            total_ms += ctx.timer_stop()
        return total_ms, out

    step_dev = lambda: pipe.run_raw(d_batch.ptr, True, B)
    for _ in range(max(args.warmup, 3)):
        last = step_dev()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = pipe.launch_count()
    wall0 = time.perf_counter()
    ms, last = timed(step_dev, args.steps)              # the headline number carries no profiling events
    barrier()
    wall = time.perf_counter() - wall0
    launches = pipe.launch_count() - l0
    clocks = sampler.stop()
    dump = result_arrays(last, S) if args.dump_outputs and rank == 0 else {}

    # ------------------------------------------------------------------ e2e: host buffers in, clouds out
    e2e = None
    if not args.no_e2e:
        lib = _cabi.load_library()
        hin, hout = C.c_void_p(), C.c_void_p()
        stride = S * P
        assert lib.kp_host_alloc(batch.nbytes, C.byref(hin)) == 0
        assert lib.kp_host_alloc(B * stride * 12, C.byref(hout)) == 0
        C.memmove(hin, batch.ctypes.data, batch.nbytes)
        step_e2e = lambda: pipe.run_host(hin.value, B, hout.value, stride)
        for _ in range(2):
            res = step_e2e()
        barrier()
        ms_e2e, res = timed(step_e2e, args.steps)
        barrier()
        d2h = sum(int(res[f].n_out) * 12 for f in range(B)) + B * C.sizeof(_cabi.FrameResult)
        e2e = {"ms": ms_e2e, "h2d": int(batch.nbytes), "d2h": int(d2h)}
        if args.dump_outputs and rank == 0:
            xyz = np.ctypeslib.as_array((C.c_float * (B * stride * 3)).from_address(hout.value)).reshape(B, stride, 3)
            dump.update(cloud_sample(xyz, [res[f].n_out for f in range(B)]))
        lib.kp_host_free(hin)
        lib.kp_host_free(hout)
    if dump:
        write_outputs(args.dump_outputs, dump)

    # ------------------------------------------------------------------ reduce over ranks (max time) before the rank-0-only legs
    per_rank = None
    if world > 1:
        # every rank's own figures travel to rank 0 (after the timed regions): the spread tells a slow GPU from a busy host
        mine = torch.tensor([ms, e2e["ms"] if e2e else 0.0, clocks.get("sm_mhz") or 0.0, 1.0 if "sw_power_cap" in clocks.get("reasons", []) else 0.0],
                            dtype=torch.float64, device="cuda")
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {"ms_per_step": [round(float(a[0]) / args.steps, 2) for a in allr],
                    "e2e_ms_per_step": [round(float(a[1]) / args.steps, 2) for a in allr],
                    "sm_mhz": [float(a[2]) for a in allr], "sw_power_cap": [bool(a[3] > 0) for a in allr]}
        t = mine[:2].clone()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e_max = float(t[0]), float(t[1])
    else:
        ms_e2e_max = e2e["ms"] if e2e else 0.0
    frames_total = world * B * args.steps
    value = frames_total / (ms * 1e-3)

    prof, prof_frames, ms_serial, c5, legs, stats = {}, 1, 0.0, None, {}, None
    if rank == 0:
        # Per-kernel durations: the same frames through ONE frame per launch, one batch at a time, as direct launches
        # with a CUDA event pair around every kernel family (profiling mode of the engine), L2 flushed between steps.
        import copy as _copy
        cfg1 = _copy.copy(cfg)
        cfg1.n_streams = fpl                 # the same frames per launch as the timed region, ONE batch in flight
        pipe1 = FramePipeline(cfg1, tab, T_fuse, T_icp, device=local_rank)
        pipe1.run_raw(d_batch.ptr, True, fpl)
        psteps = max(1, min(args.steps, 3))
        nprof = max(fpl, (min(B, 8) // fpl) * fpl)
        pipe1.profile(True)
        for _ in range(psteps):
            ctx.flush_l2(); ctx.sync(); ctx.timer_start()
            pipe1.run_raw(d_batch.ptr, True, nprof)
            ms_serial += ctx.timer_stop()
        prof = pipe1.profile_read()
        pipe1.profile(False)
        stats = pipe1.frame_counts()
        pipe1.close()
        prof_frames = nprof * psteps

        # ---------------------------------------------------------------- config C5: final clouds -> [B, 4096, 3]
        if not args.no_resample:
            n_out = [int(last[f].n_out) for f in range(B)]
            stride = S * P
            d_out = ctx.empty((B, stride, 3), np.float32)
            pipe.run_raw(d_batch.ptr, True, B, d_out_ptr=d_out.ptr, out_stride=stride)
            off = np.zeros(B + 1, np.int64)
            packed = ctx.empty((sum(n_out), 3), np.float32)
            pos = 0
            for f in range(B):
                ctx.check(ctx.lib.kp_memcpy_d2d(ctx.handle, packed.ptr + 12 * pos, d_out.ptr + 12 * f * stride, 12 * n_out[f]))
                pos += n_out[f]
                off[f + 1] = pos
            out_t = ctx.empty((B, 4096, 3), np.float32)
            fn = lambda: ctx.check(ctx.lib.kp_resample_batch(ctx.handle, packed.ptr, off.ctypes.data_as(C.POINTER(C.c_int64)), B, 4096, 0,
                                                             1234, 0, out_t.ptr, None))
            for _ in range(3):
                fn()
            ctx.sync()
            ms_c5 = 0.0
            reps = 5
            for _ in range(reps):
                ctx.flush_l2(); ctx.sync(); ctx.timer_start(); fn(); ms_c5 += ctx.timer_stop()
            c5 = {"clouds_per_s": B * reps / (ms_c5 * 1e-3), "ms_per_cloud": ms_c5 / (B * reps), "points_in": int(np.mean(n_out)),
                  "points_out": 4096, "algorithmic_GBps": round((sum(n_out) * (12 + 4 + 3 * 4) + B * 4096 * 32) * reps / (ms_c5 * 1e-3) / 1e9, 1),
                  "algorithmic_bytes": "per point 12 (row read for the key) + 4 (key write) + 3 x 4 (radix-select passes); per output 32"}
            del d_out, packed, out_t

        # ---------------------------------------------------------------- legs for BASELINE configs C1, C2, C3
        if not args.no_legs:
            from kinectpy_b200 import synth
            # C1: ONE NFOV sensor -> 1 cm voxel -> SOR(20, 2.0)
            _, d1, t1, Tf1, Ti1 = make_inputs("NFOV", 2, 0, sensors=1)
            cfgc1 = PipelineConfig(n_sensors=1, pixels=synth.NFOV.pixels, do_floor=False, do_icp=False, n_streams=16)
            p1, dd1, r1, ms1 = run_pipeline_leg(ctx, cfgc1, d1, t1, Tf1, Ti1, local_rank, 32, 3)
            legs["C1_nfov_voxel_sor"] = {"frames_per_s": round(32 / (ms1 * 1e-3), 1), "ms_per_frame": round(ms1 / 32, 4),
                                         "points": int(r1[0].n_fused), "voxels": int(r1[0].n_voxel), "kept": int(r1[0].n_sor),
                                         "workload": "1 x NFOV 640x576 -> unproject -> voxel 1 cm -> SOR(20, 2.0), 32 frames per step, depth resident"}
            p1.close(); del dd1
            # C2: 3 x NFOV fused + point-to-plane ICP of both subs (max_corr 2 cm, <= 30 iterations): ms / pair from the profile
            _, d2, t2, Tf2, Ti2 = make_inputs("NFOV", 2, 0)
            cfgc2 = PipelineConfig(n_sensors=3, pixels=synth.NFOV.pixels, n_streams=1)
            p2 = FramePipeline(cfgc2, t2, Tf2, Ti2, device=local_rank)
            dd2 = p2.upload(d2)
            p2.run_raw(dd2.ptr, True, 2)
            p2.profile(True)
            ctx.flush_l2(); ctx.sync()
            r2 = p2.run_raw(dd2.ptr, True, 2)
            pr2 = p2.profile_read()
            p2.profile(False)
            npairs = 2 * 2
            legs["C2_nfov_icp"] = {"icp_ms_per_pair": round(pr2["icp"]["ms"] / npairs, 4), "pairs": npairs,
                                   "iters": [int(r2[0].icp_iters[i]) for i in range(2)], "fitness": [round(float(r2[0].icp_fitness[i]), 4) for i in range(2)],
                                   "source_points": int(p2.frame_counts()["n_icp"][1]), "target_points": int(p2.frame_counts()["n_icp"][0]),
                                   "workload": "3 x NFOV fused; sub_i -> master on 1 cm voxel clouds, normals r = 2 cm / 30 nn, max_corr 2 cm, <= 30 it, 1e-6 / 1e-6; "
                                               "one frame (two pairs) per launch, one batch in flight: the latency of a pair, not its share of a full GPU"}
            p2.close(); del dd2
            # C3: segment_plane(1 cm, n = 3, 1000 hypotheses) on the whole fused WFOV cloud through the C ABI
            xyz = ctx.empty((S * P, 3), np.float32)
            dtab = ctx.to_device(np.ascontiguousarray(tab, np.float32), np.float32)
            Tf = np.ascontiguousarray(T_fuse, np.float64).reshape(-1)
            ctx.check(ctx.lib.kp_unproject_transform(ctx.handle, d_batch.ptr, dtab.ptr, Tf.ctypes.data, 1, S, P, cfg.unproject_flags,
                                                     float(cfg.scale), xyz.ptr, None, None, None, None))
            comp = ctx.empty((S * P, 3), np.float32)
            nfused = C.c_int64()
            ctx.check(ctx.lib.kp_compact(ctx.handle, S * P, None, 0, xyz.ptr, comp.ptr, None, None, None, None, None, C.byref(nfused)))
            plane = (C.c_double * 4)()
            ninl, best = C.c_int64(), C.c_int32()
            fn3 = lambda: ctx.check(ctx.lib.kp_ransac_plane(ctx.handle, comp.ptr, nfused.value, 0.01, 3, 1000, 0.99999999, 1234, plane, None,
                                                            C.byref(ninl), C.byref(best), None))
            for _ in range(2):
                fn3()
            ms3, reps = 0.0, 5
            for _ in range(reps):
                ctx.flush_l2(); ctx.sync(); ctx.timer_start(); fn3(); ms3 += ctx.timer_stop()
            ms3 /= reps
            props = torch.cuda.get_device_properties(local_rank)
            fp64_peak = props.multi_processor_count * 64 * 2 * 1.965e9 / 1e12      # 64 FP64 FMA lanes per SM and clock
            flops = 7.0 * nfused.value * 1000
            legs["C3_ransac_fused_wfov"] = {"ms": round(ms3, 4), "points": int(nfused.value), "hypotheses": 1000, "inliers": int(ninl.value),
                                            "fp64_tflops": round(flops / (ms3 * 1e-3) / 1e12, 2), "fp64_peak_tflops_nominal": round(fp64_peak, 1),
                                            "frac_of_fp64_peak": round(flops / (ms3 * 1e-3) / 1e12 / fp64_peak, 3),
                                            "note": "7 N H flop (3 mul + 3 add + compare per plane test, in f64 without contraction); the call includes the fit, "
                                                    "the host replay of the best / early-exit rule, the inlier mask and the refit"}
            del xyz, comp, dtab

    if rank == 0:
        peak, peak_src = peaks()
        fam = dict(prof)
        algo = family_bytes(stats, cfg, S, P, [int(x) for x in last[0].icp_iters[:S - 1]]) if stats else {}
        leaf_ms = sum(v["ms"] for k, v in fam.items() if k in LEAF) or 1.0
        table = {}
        for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"]):
            if k not in LEAF:
                continue                      # (sor / floor_sor / normals / icp_branch are scopes around their leaf families)
            per_frame_ms = v["ms"] / prof_frames
            gbs = algo.get(k, 0.0) / (per_frame_ms * 1e-3) / 1e9 if per_frame_ms > 0 else 0.0
            table[k] = {"ms_per_frame": round(per_frame_ms, 4), "share": round(v["ms"] / leaf_ms, 4), "launch_groups": v["calls"],
                        "kernel": LEAF[k][0], "bound": LEAF[k][1], "algorithmic_GBps": round(gbs, 1), "frac_of_hbm_peak": round(gbs / peak, 4)}
        top = next(iter(table), None)
        roofline = None
        if top:
            t = table[top]
            ncu = {}
            try:
                # every captured instance of the kernel (template arguments differ per k), weighted by its launches
                allk = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_summary.json")))
                inst = [v for k_, v in allk.items() if k_ == t["kernel"] or k_.startswith(t["kernel"] + "<")]
                nl = sum(v["launches"] for v in inst)
                if nl:
                    wavg = lambda key: sum(v[key] * v["launches"] for v in inst) / nl
                    ncu = {"dram_bytes_per_launch": round(wavg("dram_bytes_per_launch")), "issue_active_frac": round(wavg("issue_active_frac"), 4),
                           "warp_instructions_per_launch": round(wavg("warp_instructions_per_launch")),
                           "lanes_per_instruction": round(wavg("lanes_per_instruction"), 2), "source": inst[0]["source"],
                           "frames_per_launch": inst[0].get("frames_per_launch")}
            except Exception:
                pass
            # working launches per batch: three level-0 searches (SOR, floor SOR, normals); an ICP pass launch advances every pair
            # of the batch, and the pairs need icp_iters + 1 of the max_iter + 1 enqueued passes (the others leave at once)
            launches_per_batch = {"knn_level0": 3.0}.get(top, 1.0)
            if top == "icp":
                launches_per_batch = float(np.mean([int(last[0].icp_iters[i]) + 1 for i in range(S - 1)]))
            ach = t["algorithmic_GBps"]
            roofline = {"kernel": t["kernel"], "family": top, "bound": t["bound"], "achieved": ach, "peak": peak, "unit": "GB/s",
                        "frac": round(ach / peak, 5), "traffic": ncu.get("dram_bytes_per_launch"), "traffic_source": ncu.get("source"),
                        "traffic_frames_per_launch": ncu.get("frames_per_launch"),
                        "peak_source": peak_src, "frames_per_launch": fpl, "avg_launch_ms": round(t["ms_per_frame"] * fpl / launches_per_batch, 4),
                        "algorithmic_bytes_per_launch": round(algo.get(top, 0.0) * fpl / launches_per_batch),
                        "issue_active_frac": ncu.get("issue_active_frac"), "warp_instructions_per_launch": ncu.get("warp_instructions_per_launch"),
                        "lanes_per_instruction": ncu.get("lanes_per_instruction"),
                        "note": "dominant kernel by summed device time (CUDA events around every kernel family, one batch in flight); a launch "
                                "covers `frames_per_launch` frames. It is bound by instruction issue, not by HBM: `achieved` / `frac` are its "
                                "compulsory bytes over its run time against the HBM peak, as the contract asks; `issue_active_frac` and "
                                "`lanes_per_instruction` (ncu, profiles/) describe its real ceiling. HBM-bound families and their fractions are in `kernels`."}
        cb = None
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_baseline(cfg, depth, tab, T_fuse, T_icp, args.cpu_sample_frames)
        r0 = last[0]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config,
            "clocks": clocks, "gpu_launches": int(launches), "launches_per_frame": round(launches / max(B * args.steps, 1), 1),
            "wall_s_timed_region": round(wall, 3),
            "e2e": None if e2e is None else {"value": frames_total / (ms_e2e_max * 1e-3), "unit": UNIT,
                                             "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                                             "ms_per_step": ms_e2e_max / args.steps},
            "per_rank": per_rank,
            "roofline": roofline, "kernels": table,
            "kernels_note": "per-family device time with %d frames per launch (as in the timed region) and ONE batch in flight, CUDA events around "
                            "every family (serial ms/frame %.3f); the timed region overlaps %d such batches" % (fpl, ms_serial / prof_frames, slots),
            "cpu_baseline": cb,
            "frame_stats": {"n_fused": int(r0.n_fused), "n_voxel": int(r0.n_voxel), "n_sor": int(r0.n_sor),
                            "n_floor_inliers": int(r0.n_floor_inliers), "n_out": int(r0.n_out),
                            "icp_iters": [int(r0.icp_iters[i]) for i in range(2)],
                            "icp_fitness": [round(float(r0.icp_fitness[i]), 4) for i in range(2)],
                            # queries each level of the neighbour search hands on (SOR k=20, floor SOR k=50, normals)
                            "knn_left_after_level0": stats.get("leftovers_l0") if stats else None,
                            "knn_left_after_level1": stats.get("leftovers_l1") if stats else None,
                            "n_merged": stats.get("n_merged") if stats else None,
                            "n_icp_clouds": stats.get("n_icp") if stats else None},
        }
        icpv = fam.get("icp")
        if icpv:
            line["icp_ms_per_pair"] = round(icpv["ms"] / prof_frames / 2, 4)
            line["icp_ms_per_pair_note"] = "WFOV pair inside C4 (one frame per launch); the NFOV pair of config C2 is legs.C2_nfov_icp"
        if c5 is not None:
            line["resample_c5"] = c5
        if legs:
            line["legs"] = legs
        print(json.dumps(line))
    pipe.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
