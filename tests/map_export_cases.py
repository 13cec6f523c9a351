"""Cases of the map export (lsd_slam_viewer's KeyFrameDisplay::flushPC, lsdgpu_map_export_points): filter settings, poses,
levels and adversarial idepth / variance planes, shared by the oracle pin (tests/test_map_export_pin.py, records stored by
tests/golden/make_map_export_golden.py) and the GPU tests (tests/test_gpu_map_export.py)."""
import hashlib

import numpy as np

# (scaledDepthVarTH, absDepthVarTH, minNearSupport): the viewer's built-in defaults (settings.cpp:36-38), the ROS defaults
# (cfg/LSDSLAMViewerParams.cfg:20-22, 10^-3 / 10^-1 / 7), the near-support test off (0, 1), and at its maximum (9) under an
# absolute threshold that binds for scale != 1
FILTERS = [(1.0, 1.0, 5), (1e-3, 1e-1, 7), (1e-3, 1e-1, 0), (1.0, 1.0, 1), (1e-2, 5e-3, 9)]
LEVELS = (0, 1, 2)


def _quat(axis, angle):
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    return np.concatenate([a * np.sin(angle / 2), [np.cos(angle / 2)]])


# camToWorld as (qx, qy, qz, qw, tx, ty, tz, scale): scale 1 and two scales != 1 (a keyframe graph rescales its keyframes)
POSES = [
    np.concatenate([_quat([0.3, -0.8, 0.2], 0.7), [0.25, -1.5, 3.0], [1.0]]),
    np.concatenate([_quat([-0.5, 0.1, 0.9], 2.1), [-4.0, 0.75, 0.125], [1.7]]),
    np.concatenate([_quat([0.0, 0.0, 1.0], -0.3), [10.0, 20.0, -5.0], [0.35]]),
]


def level_cam(K, level):
    """Frame::fx/fy/cx/cy(level) as Frame::initialize computes them (Frame.cpp:403-459): fx halves per level in float,
    cx = (cx0 + 0.5) / 2^level - 0.5 in double, cast to float"""
    K = np.asarray(K, np.float32).reshape(3, 3)
    fx, fy = K[0, 0], K[1, 1]
    for _ in range(level):
        fx, fy = np.float32(np.float64(fx) * 0.5), np.float32(np.float64(fy) * 0.5)
    cx = np.float32((np.float64(K[0, 2]) + 0.5) / (1 << level) - 0.5)
    cy = np.float32((np.float64(K[1, 2]) + 0.5) / (1 << level) - 0.5)
    if level == 0:
        cx, cy = K[0, 2], K[1, 2]
    return np.array([fx, fy, cx, cy], np.float32)


def adversarial_planes(w, h, seed):
    """idepth / idepthVar planes that drive every branch of the filter: tiny (depth^4 overflows to inf), zero, negative, denormal,
    infinite and NaN values next to ordinary ones, in 3x3-coherent patches so that near support is both met and missed"""
    rng = np.random.default_rng(seed)
    base = rng.uniform(0.2, 2.0, (h // 4 + 1, w // 4 + 1)).astype(np.float32)
    idepth = np.kron(base, np.ones((4, 4), np.float32))[:h, :w].copy()
    idepth *= rng.uniform(0.97, 1.03, (h, w)).astype(np.float32)
    var = (rng.uniform(0, 1, (h, w)) ** 4 * 0.05).astype(np.float32)
    special_id = np.array([1e-30, 1e-20, 1e-12, 0.0, -0.0, -0.5, 1e-40, 1.4e-45, np.inf, -np.inf, np.nan, 3e38], np.float32)
    special_var = np.array([0.0, -0.0, 1e-40, 1e-30, np.inf, np.nan, -1.0, -2.0, 3e38, 1e-7], np.float32)
    m = rng.random((h, w))
    sel = m < 0.15
    idepth[sel] = special_id[rng.integers(0, special_id.size, int(sel.sum()))]
    sel = (m > 0.85)
    var[sel] = special_var[rng.integers(0, special_var.size, int(sel.sum()))]
    # a block of var == 0 with tiny idepth: depth^4 = inf, 0 * inf = NaN passes both thresholds
    idepth[h // 2:h // 2 + 3, w // 2:w // 2 + 3] = np.float32(1e-25)
    var[h // 2:h // 2 + 3, w // 2:w // 2 + 3] = 0
    return idepth, var


def records_from_planes(idepth, var, image):
    """keyframeMsg.pointcloud of the planes (ROSOutput3DWrapper.cpp:99-107): float image -> uchar colour"""
    from oracle import map_oracle
    rec = np.zeros(idepth.size, map_oracle.POINT_DENSE)
    rec["idepth"] = idepth.ravel()
    rec["idepth_var"] = var.ravel()
    rec["color"] = np.clip(image.ravel(), 0, 255).astype(np.uint8)[:, None]
    return rec


def points_digest(points):
    return hashlib.sha256(np.ascontiguousarray(points, np.float32).view(np.uint32).tobytes()).hexdigest()


def oracle_inputs(seq, frames, fast=False):
    """name -> (list of level records).  'gt': keyframe 0 with GT depth (Frame::setDepthFromGroundTruth); 'mapped_kf0' /
    'mapped_kf4': keyframes of a mapped run on the oracle (frames 1-4 mapped into keyframe 0, keyframe change to frame 4 with
    finalizeKeyFrame + createKeyFrame, frames 5-7 mapped into it, finalizeKeyFrame); 'adversarial': the planes above."""
    from oracle import pyoracle as po
    po.set_globals(fast)
    out = {}
    kf0 = po.Frame(0, frames[0][0], seq.K, fast=fast)
    kf0.setDepthFromGroundTruth(frames[0][1])
    out["gt"] = [kf0.pack_pointcloud(l) for l in LEVELS]
    dm = po.DepthMap(seq.w, seq.h, seq.K, fast=fast)
    dm.initializeFromGTDepth(kf0)
    settings = po.default_track_settings(fast)
    kf, last, keep = kf0, np.array([0, 0, 0, 1, 0, 0, 0], np.float64), []
    for k in range(1, 8):
        f = po.Frame(k, frames[k][0], seq.K, fast=fast)
        r = po.se3_track(kf, f, last, settings)
        last = np.array(r.frameToRef_qt)
        kf.L.lsdo_frame_set_depthHasBeenUpdatedFlag(kf.ptr, 0)
        dm.updateKeyframe([f])
        keep.append(f)
        if k == 4:
            dm.finalizeKeyFrame()
            out["mapped_kf0"] = [kf0.pack_pointcloud(l) for l in LEVELS]
            dm.createKeyFrame(f)
            kf, last = f, np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
    dm.finalizeKeyFrame()
    out["mapped_kf4"] = [kf.pack_pointcloud(l) for l in LEVELS]
    adv = []
    for l in LEVELS:
        w, h = seq.w >> l, seq.h >> l
        idepth, var = adversarial_planes(w, h, seed=100 + l)
        adv.append(records_from_planes(idepth, var, kf0.image(l)))
    out["adversarial"] = adv
    return out


def pin_records(seq, frames, flavour):
    """every (input, level, filter, pose) case run on one flavour of lsdo_map_export (False = oracle/lsd_oracle_map.c,
    "ref_viewer" = the viewer's own code): {case: {"n": points, "sha256": digest}}"""
    from oracle import map_oracle
    inputs = oracle_inputs(seq, frames)            # the records are inputs: always the C oracle's, whatever `flavour` is
    res = {}
    for name, per_level in inputs.items():
        for li, l in enumerate(LEVELS):
            cam = level_cam(seq.K, l)
            for fi, (sth, ath, mns) in enumerate(FILTERS):
                for pi, qts in enumerate(POSES):
                    pts = map_oracle.map_export(per_level[li], seq.w >> l, seq.h >> l, cam, qts, sth, ath, mns, flavour)
                    res[f"{name}/L{l}/F{fi}/P{pi}"] = {"n": int(pts.shape[0]), "sha256": points_digest(pts)}
    return res
