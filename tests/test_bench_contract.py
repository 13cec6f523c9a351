"""bench.py's reference arm runs on the host only: check the JSON contract of the line the driver parses (keys, units, the
e2e / cpu_baseline objects of the CPU arm) without a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert base["metric"].startswith(d["metric"].split(" at ")[0])           # BASELINE.json's metric, 640x480 configuration
    assert d["impl"] == "reference"
    assert d["metric"] == "frames/sec (track+depth-update) at 640x480" and d["unit"] == "frames/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config"):
        assert k in d, k
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and abs(d["value"] - 1e3 / d["ms_per_step"]) < 1e-6 * d["value"]
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    from oracle import pyoracle
    # the reference's own sources (oracle/_ref) whenever they are here, the C port otherwise
    assert cb["kind"] == ("reference" if pyoracle.ref_available() else "port")
    assert cb["cores"] == 5 and cb["value"] == d["value"] and "sample" in cb
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_bench_refuses_to_run_the_gpu_arm_without_a_gpu():
    """no CPU fallback: without a CUDA device the product arm fails loudly instead of printing a number"""
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3", "--no-cpu-baseline"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0
    assert not any(ln.strip().startswith("{") for ln in r.stdout.splitlines())


def _fake_gpu_run_factory(bench):
    import numpy as np

    def fake_gpu_run(args, rank, world, local_rank):
        n = args.warmup + args.steps
        seq, frames = bench.render_frames(args.width, args.height, 1234, n + 1)
        pr = [{"rank": 0, "sum_ms": 2.0, "p50": 0.2, "p95": 0.22, "max_step_ms": 0.3, "argmax_step": 1, "pass_ms": [2.0],
               "sm_mhz": 1965.0, "reasons": [], "pinned_cores": None}]
        leg = dict(pass_ms=[2.0], launches=53, clocks={"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": [], "samples": 5}, wall=0.1,
                   kms=1.1, klaunch=10, kbytes=1.1e8, poses=np.zeros((n, 7)), p50=0.2, p95=0.22, per_rank=pr)
        return seq, frames, {"resident": leg, "e2e": dict(leg, pass_ms=[2.2])}
    return fake_gpu_run


def _fake_parity_leg_factory(bench, pose_rel):
    def fake_parity_leg(args, seq, frames, res):
        n = min(len(frames), args.warmup + args.steps + 1)
        o = bench.cpu_loop(seq, frames[:n], n - 1, 0, time_budget_s=0, flavour=False)
        par = {"tolerance": bench.POSE_TOL, "frames": 5, "max_pose_rel": pose_rel, "maps_identical": True, "legs_bit_identical": True}
        par["ok"] = pose_rel <= bench.POSE_TOL
        return par, o["poses"]
    return fake_parity_leg


def test_product_arm_line_contract_with_mocked_device_results(monkeypatch, capsys):
    """the JSON line of the product arm (everything after the device timing): all contract keys, roofline, cpu_baseline,
    e2e, clocks, gpu_launches, the in-run parity record -- exercised on the CPU by replacing only the two device loops"""
    sys.path.insert(0, ROOT)
    import bench
    from oracle import pyoracle
    monkeypatch.setattr(bench, "gpu_run", _fake_gpu_run_factory(bench))
    monkeypatch.setattr(bench, "parity_leg", _fake_parity_leg_factory(bench, 2e-5))
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "20", "--warmup", "3"])
    bench.main()
    lines = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "clocks", "gpu_launches", "parity", "per_rank", "pass_ms"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 20 and d["gpu_launches"] == 53 and d["vs_baseline"] is None
    assert abs(d["value"] - 20 / 2.0e-3) < 1e-6 and abs(d["e2e"]["value"] - 20 / 2.2e-3) < 1e-6
    assert d["e2e"]["h2d_bytes_per_step"] == 640 * 480 and d["e2e"]["d2h_bytes_per_step"] > 0
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-12
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if pyoracle.ref_available() else "port")
    assert cb["cores"] == 5 and cb["value"] > 0 and cb["single_core"]["value"] > 0
    assert 0.30 <= d["config"]["semi_dense_fraction"] <= 0.50 and "workload" in d["config"] and "l2" in d["config"]
    par = d["parity"]
    assert par["ok"] is True and par["tolerance"] == 1e-4
    if cb["kind"] == "reference":
        assert par["reference_sse_vs_scalar"]["max_pose_rel"] > 1e-4        # the stock SSE build is NOT within 1e-4 of its scalar path


def test_product_arm_fails_when_parity_is_off(monkeypatch, capsys):
    """a pose 3e-4 away from the oracle on a replayed step: the line still prints (parity.ok false), the process exits non-zero"""
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "gpu_run", _fake_gpu_run_factory(bench))
    monkeypatch.setattr(bench, "parity_leg", _fake_parity_leg_factory(bench, 3e-4))
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "4", "--warmup", "3", "--no-cpu-baseline"])
    with pytest.raises(SystemExit) as ei:
        bench.main()
    assert ei.value.code == 3
    d = json.loads([ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")][0])
    assert d["parity"]["ok"] is False


@pytest.mark.gpu
def test_dump_outputs_are_identical_across_runs(tmp_path):
    """--dump-outputs writes the last timed step's results as float32 / float64 .npy files within 64 MB; two runs with the same
    arguments see the same seeded stream and must write the same arrays bit for bit (the kernels use no float atomics)"""
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "6", "--warmup", "3", "--width", "320", "--height", "240",
                            "--no-cpu-baseline", "--no-parity", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 6
        assert sum(p.stat().st_size for p in d.iterdir()) <= 64 << 20
        dumps.append({p.stem: np.load(p) for p in d.glob("*.npy")})
    a, b = dumps
    assert {"pose_qt", "track_result", "new_kf_thisToParent_qts", "depth_isValid", "depth_idepth", "depth_idepth_var"} <= set(a)
    assert set(a) == set(b)
    for name, x in a.items():
        assert x.dtype in (np.float32, np.float64), name
        assert x.tobytes() == b[name].tobytes(), name
    assert a["pose_qt"].shape == (7,) and np.isfinite(a["pose_qt"]).all() and a["depth_idepth"].shape == (240, 320)
    assert a["depth_isValid"].sum() > 10000
