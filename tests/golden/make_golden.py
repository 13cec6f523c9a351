"""Generates the golden vectors under tests/golden/ on the seeded 320x240 synthetic stream.

  reference_320x240.npz     OUTPUTS OF THE REFERENCE ITSELF: computed by oracle/_ref/liblsd_ref.so, i.e. by the reference's own
                            DepthMap.cpp / SE3Tracker.cpp / Sim3Tracker.cpp / TrackingReference.cpp / Frame.cpp and the vendored
                            Sophus, compiled unmodified (oracle/ref_build.py; scalar code path, strict IEEE).  The C oracle must
                            reproduce them bit for bit (tests/test_oracle_kats.py) and the CUDA path is compared with them on the
                            GPU (tests/test_gpu_golden.py).  Needs /root/reference (present in the build container only).
  oracle_8f_320x240.npz     Sim3 entries from the reference-compiled library as above; keyframeMsg packing, re-activation data and
                            UndistorterPTAM from the C oracle (their reference sources need ROS message headers / OpenCV remap and
                            are not part of oracle/_ref).
  ref_pin_320x240.json      the records of tests/test_ref_pin.py's cases computed by the reference-compiled libraries
                            (oracle/_ref/liblsd_ref.so, liblsd_ref_sse.so); the C oracle must reproduce them.
  reference_files.json      line count of every file of the reference tree, by path relative to its root: what
                            tests/test_citations.py resolves the `path:line` citations against.
The reference-generated files need the reference sources (oracle/ref_build.py builds oracle/_ref from them).
Run:  python -m tests.golden.make_golden
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
IDENT = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)


def compute(oracle, seq, frames):
    out = {}
    img0, d0 = frames[0]
    kf = oracle.Frame(0, img0, seq.K)
    kf.setDepthFromGroundTruth(d0)
    dm = oracle.DepthMap(seq.w, seq.h, seq.K)
    dm.initializeFromGTDepth(kf)
    out["input_frame0_u8_crc"] = np.array([int(img0.astype(np.uint64).sum()), int((img0.astype(np.uint64) * np.arange(img0.size).reshape(img0.shape) % 65521).sum())], np.uint64)
    out["maxgrad0_row100"] = kf.maxGradients(0)[100].copy()
    out["idepth_l2"] = kf.idepth(2).copy()
    out["idepthvar_l3"] = kf.idepthVar(3).copy()
    last = IDENT
    poses = []
    for k in range(1, 6):
        f = oracle.Frame(k, frames[k][0], seq.K)
        r = oracle.se3_track(kf, f, last)
        last = np.array(r.frameToRef_qt)
        poses.append(last)
        kf.L.lsdo_frame_set_depthHasBeenUpdatedFlag(kf.ptr, 0)
        dm.updateKeyframe([f])
        if k == 5:
            out["goodmask_f5"] = (f.refPixelWasGood() != 0).astype(np.uint8)      # bool: the reference memsets "true" as 0xFF (Frame.h:433)
            dm.createKeyFrame(f)
            out["new_kf_pose_qts"] = f.thisToParent()
    out["poses_1_5"] = np.array(poses)
    cur = dm.current()
    valid = cur["isValid"][60:180:3, 80:240:3] != 0
    for n in ("isValid", "blacklisted", "validity_counter", "idepth", "idepth_var", "idepth_smoothed", "idepth_var_smoothed"):
        a = cur[n][60:180:3, 80:240:3].copy()
        if n not in ("isValid", "blacklisted"):
            a[~valid] = 0           # never-valid pixels hold uninitialised heap memory in the reference (DepthMapPixelHypothesis.h:63-64)
        out["hyp_" + n] = a
    return out


def compute_8f(oracle, seq, frames):
    """SURVEY 8f rows: Sim3 tracking, keyframe output formats, UndistorterPTAM"""
    import zlib
    out = {}
    kfs = {}
    for k in (0, 4):
        f = oracle.Frame(k, frames[k][0], seq.K)
        f.setDepthFromGroundTruth(frames[k][1])
        kfs[k] = f
    init = np.concatenate([seq.frame_to_ref_qt(4, 0), [1.02]])
    init[4:7] += [0.01, -0.005, 0.004]
    r = oracle.sim3_track(kfs[0], kfs[4], init, 4, 1)
    out["sim3_frameToRef_qts"] = np.array(r.frameToRef_qts)
    out["sim3_hessian"] = np.array(r.lastSim3Hessian, np.float32)
    out["sim3_residuals"] = np.array([r.lastResidual, r.lastDepthResidual, r.lastPhotometricResidual, r.pointUsage,
                                      r.affineEstimation_a, r.affineEstimation_b], np.float32)
    out["sim3_calls"] = np.array([list(r.numCalcResidualCalls), list(r.numCalcWarpUpdateCalls)], np.int32)
    dm = oracle.DepthMap(seq.w, seq.h, seq.K)
    dm.initializeFromGTDepth(kfs[0])
    dm.finalizeKeyFrame()
    a, b, c = kfs[0].reactivation_data()
    out["react_var_row120"] = b[120].copy()
    out["react_validity_hist"] = np.bincount(c.ravel(), minlength=256).astype(np.int64)
    out["pointcloud_l1_crc"] = np.array([zlib.crc32(kfs[0].pack_pointcloud(1).tobytes())], np.uint64)
    u = oracle.UndistorterPTAM([0.535719308086809, 0.669566858850269, 0.493248545285398, 0.500408664348414, 0.897966326944875],
                               (seq.w, seq.h), "crop", (seq.w, seq.h))
    out["undist_K"] = u.K.copy()
    out["undist_remapX_row60"] = u.remapX[60].copy()
    out["undist_image_crc"] = np.array([zlib.crc32(u.undistort(frames[0][0]).tobytes())], np.uint64)
    return out


class Bound:
    """oracle.pyoracle with every constructor / call bound to one flavour (False = C oracle, "ref" = reference-compiled)"""

    def __init__(self, po, flavour):
        self.po, self.fl = po, flavour
        po.set_globals(flavour)

    def Frame(self, fid, img, K):
        return self.po.Frame(fid, img, K, fast=self.fl)

    def DepthMap(self, w, h, K):
        return self.po.DepthMap(w, h, K, fast=self.fl)

    def se3_track(self, kf, f, init, settings=None):
        return self.po.se3_track(kf, f, init, settings or self.po.default_track_settings(self.fl))

    def sim3_track(self, kf, f, init, start, final):
        return self.po.sim3_track(kf, f, init, start, final, self.po.default_track_settings(self.fl, main_tracker=False))

    def UndistorterPTAM(self, *a):
        return self.po.UndistorterPTAM(*a, fast=self.fl)


SIM3_KEYS = ("sim3_frameToRef_qts", "sim3_hessian", "sim3_residuals")


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    from lsd_slam_b200 import synth
    from oracle import pyoracle
    pyoracle.build()
    if not pyoracle.ref_available():
        raise SystemExit("oracle/_ref is not built and the reference sources are absent: the reference-generated fixtures cannot be regenerated")
    seq = synth.Sequence(320, 240, seed=1234)
    frames = {k: seq.render(k) for k in range(0, 6)}
    res = compute(Bound(pyoracle, "ref"), seq, frames)                 # the reference's own code
    np.savez_compressed(os.path.join(HERE, "reference_320x240.npz"), **res)
    print({k: v.shape for k, v in res.items()})
    res = compute_8f(Bound(pyoracle, False), seq, frames)
    # Sim3: take the reference-compiled numbers (the call counters are locals of the reference, so they stay the oracle's)
    kfs = {}
    b = Bound(pyoracle, "ref")
    for k in (0, 4):
        f = b.Frame(k, frames[k][0], seq.K)
        f.setDepthFromGroundTruth(frames[k][1])
        kfs[k] = f
    init = np.concatenate([seq.frame_to_ref_qt(4, 0), [1.02]])
    init[4:7] += [0.01, -0.005, 0.004]
    r = b.sim3_track(kfs[0], kfs[4], init, 4, 1)
    res["sim3_frameToRef_qts"] = np.array(r.frameToRef_qts)
    res["sim3_hessian"] = np.array(r.lastSim3Hessian, np.float32)
    res["sim3_residuals"] = np.array([r.lastResidual, r.lastDepthResidual, r.lastPhotometricResidual, r.pointUsage,
                                      r.affineEstimation_a, r.affineEstimation_b], np.float32)
    np.savez_compressed(os.path.join(HERE, "oracle_8f_320x240.npz"), **res)
    print({k: v.shape for k, v in res.items()})

    from tests import test_ref_pin
    pin_frames = {k: seq.render(k) for k in range(0, 26)}
    with open(os.path.join(HERE, "ref_pin_320x240.json"), "w") as f:
        json.dump(test_ref_pin.reference_records(seq, pin_frames), f, indent=1)

    from oracle import ref_build
    if ref_build.available():
        ref_root = os.path.dirname(ref_build.REF)
        lines = {}
        for root, _, files in os.walk(ref_root):
            for name in files:
                p = os.path.join(root, name)
                lines[os.path.relpath(p, ref_root)] = sum(1 for _ in open(p, errors="ignore"))
        with open(os.path.join(HERE, "reference_files.json"), "w") as f:
            json.dump(dict(sorted(lines.items())), f, indent=1)
