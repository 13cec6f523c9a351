"""Map export (lsdgpu_map_export_points) on N resident 640x480 keyframes with GT depth, N in {64, 256, 1024}: the working set
(12 B per pixel of the three planes, 3.7 MB per keyframe) exceeds the 126 MB L2 from N = 64 on, so every export reads HBM.

Per N: the whole call into a pinned host buffer (count pass, scan, write pass, records copied to the host) timed with CUDA events
around it after warm-up; the kernels alone (k_map_points / k_map_scan, summed from a torch.profiler trace of one call); points/s,
ms per keyframe and algorithmic bytes (12 B per pixel read + 16 B per point written) per second against the B200's 7.7 TB/s.
CPU arms on the same keyframes (on the first CPU_KF of them, reported per keyframe): lsd_slam_viewer's own flushPC
(oracle/_ref/liblsd_ref_viewer.so, one core) on the packed records, and the path without this entry point (one
lsdgpu_keyframe_pack_pointcloud call + 3.7 MB copy per keyframe, then the same filter on the host).
Prints the card's name and power limit and one JSON line.
Run:  python scripts/bench_map_export.py [--sizes 64,256,1024] [--reps 10]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lsd_slam_b200 import abi, synth  # noqa: E402

W, H, LEVEL = 640, 480, 0
FILTER = (1e-3, 1e-1, 7)                 # the ROS viewer parameters (cfg/LSDSLAMViewerParams.cfg:20-22)
CPU_KF = 16
HBM_BPS = 7.7e12


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def quiet(fn):
    """run fn with the C library's stdout (flushPC prints a line per keyframe) sent to /dev/null"""
    sys.stdout.flush()
    saved = os.dup(1)
    with open(os.devnull, "w") as dn:
        os.dup2(dn.fileno(), 1)
        try:
            return fn()
        finally:
            os.dup2(saved, 1)
            os.close(saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="64,256,1024")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    sizes = [int(s) for s in a.sizes.split(",")]
    seq = synth.Sequence(W, H, seed=1234)
    distinct = [seq.render(k) for k in range(0, 16, 2)]              # 8 rendered views, reused round-robin over the slots
    rng = np.random.default_rng(0)
    results = {"card": card(), "width": W, "height": H, "level": LEVEL, "filter": FILTER, "sizes": {}}
    for n in sizes:
        ctx = abi.Context(W, H, seq.K, device=0, max_frames=n + 1)
        for i in range(n):
            img, d = distinct[i % len(distinct)]
            ctx.upload(i, img)
            ctx.set_depth_gt(i, d)
        ids = np.arange(n, dtype=np.int32)
        q = rng.normal(size=(n, 4))
        q /= np.linalg.norm(q, axis=1, keepdims=True)
        qts = np.concatenate([q, rng.normal(size=(n, 3)), rng.uniform(0.5, 2.0, (n, 1))], axis=1)
        pts, counts = ctx.export_map(ids, qts, LEVEL, *FILTER)       # warm-up (staging allocated, pyramids built) + sizes
        total = int(pts.shape[0])
        out = torch.empty((max(total, 1), 4), dtype=torch.float32, pin_memory=True)
        import ctypes as C
        f = abi.MapFilter(*FILTER)
        tot = C.c_longlong(0)
        args = (ctx.ptr, n, ids.ctypes.data_as(C.POINTER(C.c_int)), qts.ctypes.data_as(C.POINTER(C.c_double)), LEVEL,
                C.byref(f), C.c_void_p(out.data_ptr()), total, None, C.byref(tot))
        for _ in range(2):
            ctx._ck(ctx.L.lsdgpu_map_export_points(*args))
        ms = []
        for _ in range(a.reps):
            ctx.synchronize()
            ctx.timer_begin(0)
            ctx._ck(ctx.L.lsdgpu_map_export_points(*args))
            ctx.timer_end(0)
            ms.append(ctx.timer_ms(0))
        assert np.asarray(out[:total]).tobytes() == pts.tobytes()
        # kernels only: one call under the profiler
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx._ck(ctx.L.lsdgpu_map_export_points(*args))
            torch.cuda.synchronize()
        kern = {}
        for e in prof.events():
            if "k_map_" in e.name and e.device_type.name == "CUDA":
                key = "scan" if "scan" in e.name else ("write" if ("ILb1E" in e.name or "<true>" in e.name) else "count")
                kern[key] = kern.get(key, 0.0) + e.device_time / 1e3
        kern_ms = sum(kern.values())
        px = (W >> LEVEL) * (H >> LEVEL)
        alg_bytes = 12.0 * px * n + 16.0 * total
        call_ms = float(np.median(ms))
        r = {"keyframes": n, "points": total, "call_ms_median": call_ms, "call_ms_min": float(np.min(ms)),
             "kernel_ms": kern_ms, "kernel_ms_by_pass": kern,
             "ms_per_keyframe_call": call_ms / n, "points_per_s_call": total / (call_ms / 1e3),
             "alg_bytes": alg_bytes, "alg_bytes_per_s_kernels": alg_bytes / (kern_ms / 1e3) if kern_ms else None,
             "hbm_fraction_kernels": (alg_bytes / (kern_ms / 1e3)) / HBM_BPS if kern_ms else None,
             "alg_bytes_per_s_call": alg_bytes / (call_ms / 1e3)}
        # CPU arms on the first CPU_KF keyframes
        m = min(CPU_KF, n)
        from oracle import map_oracle
        from tests import map_export_cases as mc
        cam = mc.level_cam(seq.K, LEVEL)
        recs = [ctx.pack_pointcloud(i, LEVEL) for i in range(m)]
        if os.path.exists(map_oracle.VIEWER_LIB):
            t0 = time.perf_counter()
            quiet(lambda: [map_oracle.map_export(recs[i], W, H, cam, qts[i], *FILTER, "ref_viewer") for i in range(m)])
            r["cpu_viewer_flushPC_ms_per_keyframe"] = (time.perf_counter() - t0) * 1e3 / m
        else:
            r["cpu_viewer_flushPC_ms_per_keyframe"] = "not measured (oracle/_ref/liblsd_ref_viewer.so not built)"
        t0 = time.perf_counter()
        got = []
        for i in range(m):
            rec = ctx.pack_pointcloud(i, LEVEL)
            got.append(map_oracle.map_export(rec, W, H, cam, qts[i], *FILTER))
        r["cpu_pack_copy_filter_ms_per_keyframe"] = (time.perf_counter() - t0) * 1e3 / m
        assert np.concatenate(got).tobytes() == pts[:int(counts[:m].sum())].tobytes()
        r["speedup_call_vs_pack_copy_filter"] = r["cpu_pack_copy_filter_ms_per_keyframe"] / r["ms_per_keyframe_call"]
        results["sizes"][str(n)] = r
        ctx.close()
        del out
        print(f"N={n}: {total} points, call {call_ms:.3f} ms, kernels {kern_ms:.3f} ms", file=sys.stderr)
    results["card"] = card()
    print(json.dumps(results))


if __name__ == "__main__":
    main()
