#!/usr/bin/env python
"""bench.py -- frames/sec of the LSD-SLAM hot path (SE3Tracker::trackFrame + DepthMap::updateKeyframe, with a
forced finalizeKeyFrame + createKeyFrame every 20 frames) on a synthetic 640x480 grayscale stream.

  python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path (one stream per GPU)
  python bench.py ... --dump-outputs DIR                    # also write what the last timed step computed, DIR/<name>.npy
  python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU code (oracle/_ref, ENABLE_SSE build,
                                                            # 1 tracking + 4 mapping threads); the C port if _ref is absent

One "step" = one frame through {Frame construction, trackFrame, mapping}.  `value` is measured with the raw u8 frames already
parked in HBM (prefetch ring); `e2e` is the same loop fed from HOST buffers through the C ABI with the H2D copy of every frame
and the D2H read of the tracking result inside the timed region.

Timing: W warm-up steps, then ONE pass of EXACTLY K timed steps on consecutive fresh frames of the stream, per leg; the pass
is bracketed by barrier + synchronize, its time is the sum of the K per-step CUDA-event times (L2 flushed between steps), MAX
over ranks.  Parity is asserted in the same run (world size 1, outside the timed region): a sample of the loop's steps is replayed on the
CPU oracle from the device's own state (identical inputs); the line carries `parity` and the run fails above 1e-4.
Prints ONE JSON line on rank 0.

--dump-outputs DIR: after the timed steps, rank 0 writes what the resident leg's LAST timed step returned to its caller, so
that two builds run with the same arguments (hence the same seeded input stream) can be compared output for output:
    pose_qt.npy                        float64 [7]   frameToRef (qx, qy, qz, qw, tx, ty, tz) of the tracked frame
    track_result.npy                   float64 [20]  the other fields of lsdgpu_track_result, in the order of TRACK_FIELDS
    new_kf_thisToParent_qts.npy        float64 [8]   the new keyframe's Sim3 output of the call (set on a keyframe change)
    depth_<field>.npy                  float32 [h, w] every field of the current keyframe's depth map (lsdgpu_depth_download)
The depth map is ~10 MB at 640x480; above DUMP_BUDGET the fields hold a fixed seeded sample of the pixels instead, flattened,
and depth_sample_index.npy (float64) holds the row-major pixel index of each sampled entry.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/sec (track+depth-update) at 640x480"
KF_EVERY = 20
POSE_TOL = 1e-4           # north_star: SE3 pose within 1e-4 rel on translation / rotation
DUMP_BUDGET = 64 << 20    # bytes written by --dump-outputs at most
TRACK_FIELDS = ("pointUsage", "lastGoodCount", "lastBadCount", "lastMeanRes", "lastResidual", "affineEstimation_a",
                "affineEstimation_b", "diverged", "trackingWasGood", "numCalcResidualCalls", "numCalcWarpUpdateCalls",
                "initialTrackedResidual")


def rank_world():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def step_outputs(gs) -> dict:
    """what GpuStream.step / lsdgpu_track_and_map handed back on the last step, plus the current keyframe's depth map"""
    from lsd_slam_b200.abi import HYP_DTYPE
    r = gs.tracker.last
    out = {"pose_qt": np.array(gs.poses[-1], np.float64),
           "track_result": np.concatenate([np.ravel(getattr(r, f)) for f in TRACK_FIELDS]).astype(np.float64),
           "new_kf_thisToParent_qts": np.array(gs._qts, np.float64)}
    hyp = gs.map.current()
    fields = [f for f in HYP_DTYPE.names if f != "_pad"]
    budget = (DUMP_BUDGET - (64 << 10)) // (4 * len(fields) + 8)          # pixels that fit, with their sample index; 64 KB for the rest
    if hyp.size > budget:
        idx = np.sort(np.random.default_rng(0).choice(hyp.size, budget, replace=False))
        hyp = hyp.reshape(-1)[idx]
        out["depth_sample_index"] = idx.astype(np.float64)
    for f in fields:
        out["depth_" + f] = hyp[f].astype(np.float32)
    return out


def write_outputs(d: str, outputs: dict):
    os.makedirs(d, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(d, name + ".npy"), a)


def nvml_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        parts = vis.split(",")
        if local_rank < len(parts) and parts[local_rank].strip().isdigit():
            return int(parts[local_rank])
    return local_rank


def pin_to_gpu_numa_node(local_rank: int):
    """bind this rank to the host cores next to its GPU (NVML ideal CPU affinity = the GPU's NUMA node): on a 2-socket host
    an unpinned rank's polling thread can sit across the socket link from its GPU.  Returns the number of cores or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(nvml_index(local_rank))
        n = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cores = [64 * i + b for i, word in enumerate(mask) for b in range(64) if (word >> b) & 1]
        cores = [c for c in cores if c in os.sched_getaffinity(0)]
        if cores:
            os.sched_setaffinity(0, cores)
            return len(cores)
    except Exception:
        pass
    return None


class ClockSampler:
    """SM clocks and throttle reasons sampled DURING the timed passes (NVML every 20 ms from a thread)."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self.t = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:      # pragma: no cover
            self.err = repr(e)
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                return
            self._stop.wait(0.02)

    def stop(self):
        self._stop.set()
        if self.t:
            self.t.join(timeout=1)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [self.err or "no samples"], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def render_frames(w, h, seed, n):
    from lsd_slam_b200 import synth
    seq = synth.Sequence(w, h, seed=seed)
    frames = [seq.render(k) for k in range(n)]
    seq.density = synth.semi_dense_fraction(frames[0][0])          # SURVEY 8d: report it, refuse unrepresentative streams
    if not 0.30 <= seq.density <= 0.50:
        raise SystemExit(f"synthetic stream: maxGrad >= 5 on {100 * seq.density:.1f} % of the pixels (expected 30-50 %)")
    return seq, frames


# ------------------------------------------------------------------------------------------------------------
# CPU arm
# ------------------------------------------------------------------------------------------------------------
def cpu_flavour():
    """(flavour, kind, description): the reference's own sources (oracle/_ref, stock ENABLE_SSE build) when they are
    here, else the oracle's restatement of the same SSE loops"""
    from oracle import pyoracle as po
    if po.ref_available():
        return "ref_sse", "reference", ("lsd_slam_core's own DepthMap.cpp / SE3Tracker.cpp / Frame.cpp compiled unmodified "
                                        "(oracle/_ref, -DENABLE_SSE -O3 -march=x86-64-v3)")
    return True, "port", "oracle/lsd_oracle.c -O3 (its restatement of the reference's SSE tracker loops)"


def cpu_loop(seq, frames, n_steps, warmup, time_budget_s=25.0, multi_threading=1, flavour=None, kf_every=KF_EVERY):
    """Returns dict(fps, ms, n, threads, poses, kind, what).  Same loop as lsd_slam_b200/stream.py (oracle/cpu_stream.py).
    multi_threading=0: the reference's single-threaded fallback (IndexThreadReduce.h:72-77), i.e. one busy core."""
    from oracle import pyoracle as po
    from oracle.cpu_stream import CpuStream
    po.build()
    fl, kind, what = cpu_flavour() if flavour is None else (flavour, "port", "oracle/lsd_oracle.c, strict IEEE scalar path")
    if fl is True:
        po.set_globals(True, useSSE=1, multiThreading=multi_threading)
    else:
        po.set_globals(fl, multiThreading=multi_threading)
    cs = CpuStream(seq, fl, kf_every=kf_every)
    cs.init_gt(0, frames[0][0], frames[0][1])
    times = []
    t_begin = time.perf_counter()
    for k in range(1, len(frames)):
        _, dt = cs.step(k, frames[k][0])
        if k > warmup:
            times.append(dt)
        if len(times) >= n_steps or (time_budget_s and (time.perf_counter() - t_begin) > time_budget_s):
            break
    total = float(np.sum(times))
    return dict(fps=len(times) / total, ms=1e3 * total / len(times), n=len(times), threads=(1 + 4) if multi_threading else 1,
                poses=np.array(cs.poses), kind=kind, what=what)


def pose_errors(a, b):
    """per-frame (relative translation error, rotation angle error [rad]) between two pose lists (qx,qy,qz,qw,t)"""
    a, b = np.asarray(a), np.asarray(b)
    n = min(len(a), len(b))
    dt = np.linalg.norm(a[:n, 4:7] - b[:n, 4:7], axis=1) / np.maximum(np.linalg.norm(b[:n, 4:7], axis=1), 1e-12)
    d = np.abs(np.sum(a[:n, :4] * b[:n, :4], axis=1))
    ang = 2 * np.arccos(np.minimum(1.0, d))
    return dt, ang


def parity_leg(args, seq, frames, res):
    """Parity asserted in the same run (SURVEY 8d), OUTSIDE the timed region.

    (1) Single-step parity from the device's own state (oracle/replay.py): the loop of the timed legs is run once more and,
        for a sample of its steps (every 5th and every keyframe change), the CPU oracle -- bit-identical to the reference's
        own sources compiled without ENABLE_SSE, tests/test_ref_pin.py -- replays the same step from the same inputs: pose
        <= 1e-4 relative, depth map bit for bit with the device's pose handed over (2e-5 at a keyframe change).
    (2) The three runs of the loop (resident leg, e2e leg, this one) must have produced identical poses: the kernels
        are deterministic (no float atomics).
    (3) For information: the closed-loop distance to the oracle's own run of the loop (each side consuming its own poses).
        It is NOT bounded by 1e-4 -- the reference's mapper schedules observations on float low-order bits, so the
        reference itself drifts from a copy of itself whose poses are perturbed by 1e-6 (DESIGN.md section 5)."""
    from oracle.replay import run_with_replay
    K = args.steps
    n = min(len(frames), args.warmup + K + 1)
    sample = set(range(1, n, 5)) | {k for k in range(1, n) if k % KF_EVERY == 0}
    reps = run_with_replay(seq, frames, n, kf_every=KF_EVERY, sample=sample, mode=args.mode)
    worst = max(reps, key=lambda r: r["pose_rel"] - r["ref_noise_rel"])
    par = {"method": "single-step replay of the device's own steps on the CPU oracle (identical inputs), oracle/replay.py",
           "against": "CPU oracle, scalar path (= the reference's sources compiled without ENABLE_SSE, bit for bit)",
           "tolerance": POSE_TOL, "frames": len(reps), "keyframe_changes": int(sum(r["kf_change"] for r in reps)),
           "max_pose_rel": float(max(r["pose_rel"] for r in reps)), "median_pose_rel": float(np.median([r["pose_rel"] for r in reps])),
           "max_excess_over_reference_noise": float(worst["pose_rel"] - worst["ref_noise_rel"]), "argmax_frame": int(worst["frame"]),
           "reference_summation_noise": {"max": float(max(r["ref_noise_rel"] for r in reps)), "median": float(np.median([r["ref_noise_rel"] for r in reps])),
                                         "what": "oracle (sequential fp32 sums, = the reference) vs the same tracking with exact sums, same steps"},
           "max_pose_rel_vs_exact_sums": float(max(r["pose_rel_exact"] for r in reps)),
           "max_rot_rad": float(max(r["rot_rad"] for r in reps)),
           "lm_call_counts_equal": int(sum(r["counts_equal"] for r in reps)),
           "maps_identical": bool(all(r["map_ok"] for r in reps)),
           "max_rescale_rel": float(max([r.get("rescale_rel", 0.0) for r in reps]))}
    pr, pe = res["resident"]["poses"], res["e2e"]["poses"]
    par["legs_bit_identical"] = bool(np.array_equal(pr, pe))
    o = cpu_loop(seq, frames[:n], n - 1, 0, time_budget_s=0, flavour=False)
    dt, ang = pose_errors(pr[: n - 1], o["poses"][: n - 1])
    first_kf = min(KF_EVERY - 1, len(dt))
    par["closed_loop"] = {"frames": int(len(dt)), "max_pose_rel_before_first_keyframe_change": float(dt[:first_kf].max()),
                          "max_pose_rel": float(dt.max()), "note": "informational; see parity_leg docstring"}
    # pose tolerance: 1e-4, plus -- per step -- the reference's own summation noise on that step (see oracle/replay.py)
    par["ok"] = bool(par["max_excess_over_reference_noise"] <= POSE_TOL and par["maps_identical"] and par["legs_bit_identical"])
    return par, o["poses"]


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
def gpu_run(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from lsd_slam_b200 import abi
    from lsd_slam_b200.stream import GpuStream

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    pinned_cores = pin_to_gpu_numa_node(local_rank)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("NCCL_DEBUG", "WARN")       # keep NCCL's version banner out of stdout (one JSON line)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sync_t = torch.zeros(1, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def settle_collectives():
        """the communicator's FIRST collectives (connection set-up, proxy threads) happen here, before any warm-up or
        timed frame of a leg -- not right in front of the timed window (round 1's N = 8 outlier)"""
        if world > 1:
            for _ in range(3):
                dist.all_reduce(sync_t)
                dist.barrier()
        torch.cuda.synchronize()

    w, h = args.width, args.height
    K, W = args.steps, args.warmup
    n_frames = W + K + 1
    # independent streams: one per GPU, seeds 1234 + 1000*rank (SURVEY 8d, config 4)
    seq, frames = render_frames(w, h, 1234 + 1000 * rank, n_frames)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    # e2e leg: every frame sits in page-locked host memory (as a camera driver's DMA buffer would)
    pinned = [torch.from_numpy(f[0]).pin_memory() for f in frames]
    pinned_np = [t.numpy() for t in pinned]

    results = {}
    for leg in ("resident", "e2e"):
        ctx = abi.Context(w, h, seq.K, device=local_rank, max_frames=8)
        if leg == "resident":
            ctx.stage_reserve(n_frames)
            for k in range(n_frames):
                ctx.stage_put(k, frames[k][0])
        gs = GpuStream(ctx, mode=args.mode, kf_every=KF_EVERY)
        gs.init_gt(0, frames[0][0], frames[0][1])
        settle_collectives()
        for k in range(1, W + 1):
            gs.step(k, pinned_np[k]) if leg == "e2e" else gs.step(k, stage_index=k)
        ctx.synchronize()
        ctx.track_kernel_stats(reset=1)
        sampler = ClockSampler(nvml_index(local_rank))
        sampler.start()
        launches0 = ctx.launch_count()
        step_ms = []
        barrier()
        wall0 = time.perf_counter()
        for k in range(W + 1, W + 1 + K):
            flush.fill_(k & 0xff)                                              # L2 flush between timed steps
            torch.cuda.synchronize()
            ctx.timer_begin(0)
            if leg == "e2e":
                gs.step(k, pinned_np[k])                                       # pinned host u8 in, pose (D2H) out
            else:
                gs.step(k, stage_index=k)
            ctx.timer_end(0)
            ms = ctx.timer_ms(0)
            step_ms.append(ms)
        barrier()
        wall = time.perf_counter() - wall0
        pass_ms = [float(np.sum(step_ms))]
        clocks = sampler.stop()
        launches = ctx.launch_count() - launches0
        kms, klaunch, kbytes = ctx.track_kernel_stats(reset=2)
        t = torch.tensor(pass_ms, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                          # per pass: the slowest rank
        pass_max = [float(x) for x in t.tolist()]
        sm = np.array(step_ms)
        mine = {"rank": rank, "sum_ms": float(sm.sum()), "p50": float(np.median(sm)), "p95": float(np.percentile(sm, 95)),
                "max_step_ms": float(sm.max()), "argmax_step": int(sm.argmax()), "pass_ms": [float(x) for x in pass_ms],
                "sm_mhz": clocks.get("sm_mhz"), "reasons": clocks.get("reasons"), "pinned_cores": pinned_cores}
        per_rank = [mine]
        if world > 1:
            gathered = [None] * world
            dist.all_gather_object(gathered, mine)
            per_rank = gathered
        results[leg] = dict(pass_ms=pass_max, launches=launches, clocks=clocks, wall=wall, kms=kms, klaunch=klaunch, kbytes=kbytes,
                            poses=np.array(gs.poses), p50=float(np.median(sm)), p95=float(np.percentile(sm, 95)), per_rank=per_rank)
        if leg == "resident" and args.dump_outputs and rank == 0:
            write_outputs(args.dump_outputs, step_outputs(gs))
        ctx.close()
    return seq, frames, results


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--mode", type=int, default=1, help="tracker: 1 = device-resident LM, 0 = host-driven LM")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run parity check (profiling runs only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank, world, local_rank = rank_world()
    metric = METRIC if (args.width, args.height) == (640, 480) else METRIC.replace("640x480", f"{args.width}x{args.height}")
    workload = f"synthetic {args.width}x{args.height} grayscale stream, full track+map loop, forced keyframe every {KF_EVERY} frames"
    config = {"workload": workload, "width": args.width, "height": args.height, "pyramid_levels_tracked": "L4..L1",
              "kf_every": KF_EVERY, "streams_per_gpu": 1, "parallelism": f"{world} independent stream(s), one per GPU, no collective",
              "l2": "flushed between timed steps (256 MiB fill); per-step CUDA-event times summed",
              "passes": 1, "statistic": f"one pass of exactly {args.steps} steps (max over ranks)",
              "init": "gtDepthInit (SlamSystem.cpp:831-854)",
              "e2e_input": "one 8-bit frame per step in page-locked host memory, copied H2D inside the timed step; result block read back per step"}

    if args.impl == "reference":
        if rank != 0:
            return
        n_frames = args.warmup + args.steps + 1
        seq, frames = render_frames(args.width, args.height, 1234, n_frames)
        config["semi_dense_fraction"] = round(seq.density, 4)
        config["passes"], config["statistic"] = 1, f"mean over {args.steps} steps (wall clock, CPU)"
        c = cpu_loop(seq, frames, args.steps, args.warmup, time_budget_s=150.0)
        c1 = cpu_loop(seq, frames, min(args.steps, 30), args.warmup, time_budget_s=40.0, multi_threading=0)
        line = {"impl": "reference", "metric": metric, "value": c["fps"], "unit": "frames/s", "n_gpus": args.gpus, "steps": c["n"],
                "warmup": args.warmup, "ms_per_step": c["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": c["fps"], "unit": "frames/s", "cores": c["threads"], "kind": c["kind"],
                                 "sample": f"{c['n']} frames of the same stream; {c['what']}; 1 tracking thread + 4 mapping threads "
                                           "(MAPPING_THREADS, util/settings.h:94) as the reference threads it",
                                 "host_cores": os.cpu_count(),
                                 "single_core": {"value": c1["fps"], "unit": "frames/s", "sample": f"{c1['n']} frames, multiThreading = false"}},
                "e2e": {"value": c["fps"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    seq, frames, res = gpu_run(args, rank, world, local_rank)
    config["semi_dense_fraction"] = round(seq.density, 4)          # maxGrad >= 5 fraction of this rank's frame 0 (SURVEY 8d)
    if world > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()
    if rank != 0:
        return
    import torch  # noqa: F401
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured (MEASURED_PEAKS.json, copy burst)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    r, e = res["resident"], res["e2e"]
    K = args.steps
    pass_r, pass_e = r["pass_ms"][0], e["pass_ms"][0]
    fps = world * K / (pass_r * 1e-3)
    fps_e2e = world * K / (pass_e * 1e-3)
    traffic = None
    try:        # DRAM bytes per launch of the tracking kernel from the committed ncu --set full capture (640x480 only)
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["k_track_persistent"]
        if (args.width, args.height) == (640, 480):
            traffic = tj["dram_bytes_per_launch"]
    except Exception:
        pass
    ach = (r["kbytes"] / max(r["klaunch"], 1)) / (r["kms"] * 1e-3 / max(r["klaunch"], 1)) / 1e9 if r["kms"] > 0 else 0.0
    total_r = float(np.sum([p["sum_ms"] for p in r["per_rank"] if p["rank"] == 0]))
    line = {"metric": metric, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": pass_r / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config,
            "clocks": r["clocks"],
            "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": args.width * args.height,
                    "d2h_bytes_per_step": 144, "ms_per_step": pass_e / K, "pass_ms": e["pass_ms"]},
            "gpu_launches": int(r["launches"]),
            "pass_ms": r["pass_ms"],
            "step_ms": {"p50": r["p50"], "p95": r["p95"], "wall_ms_per_step_incl_flush": 1e3 * r["wall"] / K},
            "per_rank": r["per_rank"], "per_rank_e2e": e["per_rank"],
            "roofline": {"kernel": "warp/residual/JtJ (SE3 tracking) kernel", "bound": "hbm", "achieved": ach, "peak": hbm_peak,
                         "unit": "GB/s", "frac": ach / hbm_peak, "traffic": traffic, "peak_kind": peak_kind,
                         "share_of_step": r["kms"] / max(total_r, 1e-9),
                         "launches": int(r["klaunch"]), "avg_launch_us": 1e3 * r["kms"] / max(r["klaunch"], 1),
                         "algorithmic_bytes_per_launch": r["kbytes"] / max(r["klaunch"], 1),
                         "algorithmic_bytes": "SURVEY 8d B_fused: per evaluation 20 B per valid point + 16 B per texel of the gradient level"
                                              " (+5 B per point on L1) + 160 B, summed over the evaluations of the launch",
                         "note": "working set (<= 2.2 MB per level) is L2/SMEM resident: the kernel is latency-bound, not HBM-bound"},
            "tracker_mode": args.mode}
    failed = None
    o_poses = None
    if world == 1 and not args.no_parity:
        par, o_poses = parity_leg(args, seq, frames, res)
        line["parity"] = par
        if not par["ok"]:
            failed = f"parity: pose error {par['max_pose_rel']:.3e} (tolerance {POSE_TOL}), depth maps identical: {par['maps_identical']}"
    if not args.no_cpu_baseline and world == 1:
        n_cpu = min(len(frames) - 1 - args.warmup, K)
        c = cpu_loop(seq, frames, n_cpu, args.warmup, time_budget_s=25.0)
        c1 = cpu_loop(seq, frames, min(n_cpu, 30), args.warmup, time_budget_s=20.0, multi_threading=0)
        line["cpu_baseline"] = {"value": c["fps"], "unit": "frames/s", "cores": c["threads"], "kind": c["kind"], "ms_per_step": c["ms"],
                                "sample": f"{c['n']} frames of the same stream; {c['what']}; 1 tracking thread + 4 mapping threads",
                                "host_cores": os.cpu_count(),
                                "single_core": {"value": c1["fps"], "unit": "frames/s", "sample": f"{c1['n']} frames, multiThreading = false"}}
        if o_poses is not None and c["kind"] == "reference":
            # how far the stock (SSE) build of the reference is from its own scalar path on this stream, closed loop (DESIGN.md section 2)
            dt, ang = pose_errors(c["poses"], o_poses[: len(c["poses"])])
            line["parity"]["reference_sse_vs_scalar"] = {"max_pose_rel": float(dt.max()), "median_pose_rel": float(np.median(dt)), "frames": int(len(dt))}
    print(json.dumps(line))
    if failed:
        sys.stderr.write(failed + "\n")
        sys.exit(3)


if __name__ == "__main__":
    main()
