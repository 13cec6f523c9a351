"""Short run of every kernel for compute-sanitizer (memcheck / racecheck): 160x112 stream, keyframe change included."""
import os, sys, numpy as np
sys.path.insert(0, os.getcwd())
from lsd_slam_b200 import abi, synth
from lsd_slam_b200.stream import GpuStream
seq = synth.Sequence(160, 112, seed=7)
fr = [seq.render(k) for k in range(8)]
for mode in (1, 0):
    ctx = abi.Context(160, 112, seq.K, max_frames=8)
    gs = GpuStream(ctx, mode=mode, kf_every=4, fused_call=(mode == 1))
    gs.init_gt(0, fr[0][0], fr[0][1])
    for k in range(1, 8):
        gs.step(k, fr[k][0])
    gs.map.current(); gs.map.integral()
    ctx.download(gs.kf_id, abi.BUF_GOODMASK); ctx.depth_stats(gs.kf_id)
    ctx.close()
print("sanitize run ok")

# round 2: the sequential-sum kernels on adversarial data, and updateKeyframe with a frame tracked on another keyframe
ctx = abi.Context(160, 112, seq.K, max_frames=8)
rng = np.random.default_rng(3)
x = (rng.integers(1, 64, 70001) * 2.0 ** -9).astype(np.float32)
x[[5, 4000, 69999]] = [-1.0, np.inf, 0.0]
ctx.seq_sum_f32(x, rng.random(70001) < 0.7)
ctx.seq_sum_f32(np.full(3000, 100.0, np.float32))
ctx.upload(0, fr[0][0]); ctx.set_depth_gt(0, fr[0][1])
dm = abi.DepthMap(ctx); dm.initializeFromGTDepth(0)
for k in (1, 5):
    ctx.upload(k, fr[k][0]); ctx.set_pose(k, np.concatenate([seq.frame_to_ref_qt(k), [1.0]]), 0, 0.0)
dm.updateKeyframe([1])
dm.finalizeKeyFrame(); q5 = dm.createKeyFrame(5)
dm.updateKeyframe([(1, np.array([0, 0, 0, 1, 0.01, 0, 0, 1.0]))])
ctx.close()
print("sanitize run (round 2) ok")

# SURVEY 8f rows: permaRef batch, Sim3 batch (every cluster size), undistorter, keyframe output
import os
ctx = abi.Context(160, 112, seq.K, max_frames=8)
for k in (0, 3, 6):
    ctx.upload(k, fr[k][0]); ctx.set_depth_gt(k, fr[k][1])
se3 = abi.SE3Tracker(ctx)
ident = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)
for k in (0, 3):
    se3.setPermaRef(k)
se3.checkPermaRefOverlap([0, 3], np.array([ident, ident]))
se3.trackFrameOnPermaref([0, 3], 6, np.array([ident, ident]))
s3 = abi.Sim3Tracker(ctx)
pairs = [(0, 3), (3, 0), (0, 6), (6, 3)]
inits = np.array([np.concatenate([seq.frame_to_ref_qt(b, a), [1.01]]) for a, b in pairs])
for cs in (1, 2, 4, 8):
    os.environ["LSDGPU_SIM3_CLUSTER"] = str(cs)
    s3.trackFrameSim3Batch([p[0] for p in pairs], [p[1] for p in pairs], inits, 3, 1)
del os.environ["LSDGPU_SIM3_CLUSTER"]
s3.eval(0, 3, 2, inits[0])
dm = abi.DepthMap(ctx)
dm.initializeFromGTDepth(0)
dm.finalizeKeyFrame()
ctx.reactivation_data(0); ctx.pack_pointcloud(0, 0); ctx.pack_pointcloud(0, 2)
dm.reset(); dm.setFromExistingKF(0)
u = abi.UndistorterPTAM([0.54, 0.67, 0.49, 0.5, 0.9], (192, 128), "crop", (160, 112))
ctx2 = abi.Context(160, 112, u.getK(), max_frames=4)
u.install(ctx2)
raw = np.random.default_rng(1).integers(0, 256, (128, 192)).astype(np.uint8)
ctx2.undistort(raw); ctx2.upload_distorted(0, raw)
ctx2.close(); ctx.close()
print("sanitize run (8f rows) ok")

# map export (lsdgpu_map_export_points): count, scan and write kernels over more keyframes than one staging chunk, levels 0-2
ctx = abi.Context(160, 112, seq.K, max_frames=8)
for k in (0, 3, 6):
    ctx.upload(k, fr[k][0]); ctx.set_depth_gt(k, fr[k][1])
ids = [0, 3, 6] * 4
qts = np.array([np.concatenate([seq.frame_to_ref_qt(k), [1.0 + 0.1 * i]]) for i, k in enumerate(ids)])
for lvl in (0, 1, 2):
    ctx.export_map(ids, qts, lvl, 1.0, 1.0, 5)
    ctx.export_map(ids, qts, lvl)
ctx.close()
print("sanitize run (map export) ok")
