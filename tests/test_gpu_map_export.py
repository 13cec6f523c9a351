"""GPU map export (lsdgpu_map_export_points / abi.Context.export_map): lsd_slam_viewer's KeyFrameDisplay::flushPC
(KeyFrameDisplay.cpp:269-340) over many resident keyframes in one device pass.  The device's records must be byte-identical to
the C oracle's lsdo_map_export (pinned to the viewer's own code by tests/test_map_export_pin.py) run on the device's own packed
keyframeMsg records (lsdgpu_keyframe_pack_pointcloud) with the same poses."""
import ctypes as C

import numpy as np
import pytest

from lsd_slam_b200 import abi
from oracle import map_oracle
from tests import map_export_cases as mc

pytestmark = pytest.mark.gpu

IDENT = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)


@pytest.fixture(scope="module")
def mapped(seq_small, frames_small):
    """a device run with a keyframe change: GT init on frame 0, frames 1-4 tracked and mapped, keyframe 4 created, frames 5-7
    mapped into it; plus frame 9 with adversarial planes (lsdgpu_frame_set_idepth), frame 10 with GT depth, frame 11 without depth"""
    seq = seq_small
    ctx = abi.Context(seq.w, seq.h, seq.K, device=0, max_frames=16)
    img0, d0 = frames_small[0]
    ctx.upload(0, img0)
    ctx.set_depth_gt(0, d0)
    dm = abi.DepthMap(ctx)
    dm.initializeFromGTDepth(0)
    trk = abi.SE3Tracker(ctx, mode=1)
    trk.importFrame(0)
    kf, last = 0, IDENT
    for k in range(1, 8):
        ctx.upload(k, frames_small[k][0])
        last = trk.trackFrame(kf, k, last)
        dm.updateKeyframe([k])
        if k == 4:
            dm.finalizeKeyFrame()
            dm.createKeyFrame(4)
            kf, last = 4, IDENT
            trk.importFrame(4)
    dm.finalizeKeyFrame()
    ctx.upload(9, frames_small[9][0])
    idepth, var = mc.adversarial_planes(seq.w, seq.h, seed=7)
    ctx.set_idepth(9, idepth, var)
    ctx.upload(10, frames_small[10][0])
    ctx.set_depth_gt(10, frames_small[10][1])
    ctx.upload(11, frames_small[11][0])
    yield ctx
    ctx.close()


KFS = [0, 4, 9, 10]


def _oracle(ctx, seq, ids, poses, level, flt):
    pts, counts = [], []
    for i, q in zip(ids, poses):
        rec = ctx.pack_pointcloud(i, level)
        p = map_oracle.map_export(rec, seq.w >> level, seq.h >> level, mc.level_cam(seq.K, level), q, *flt)
        pts.append(p)
        counts.append(p.shape[0])
    return np.concatenate(pts), np.array(counts, np.int32)


def _same_bits(a, b):
    """bit-identical, except that any NaN equals any NaN (the payload of a NaN is not part of the result)"""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool((na == nb).all() and (a.view(np.uint32)[~na] == b.view(np.uint32)[~nb]).all())


@pytest.mark.parametrize("level", mc.LEVELS)
def test_export_matches_oracle(mapped, seq_small, level):
    poses = [mc.POSES[i % len(mc.POSES)] for i in range(len(KFS))]
    nan_seen = False
    for flt in mc.FILTERS:
        got, counts = mapped.export_map(KFS, poses, level, *flt)
        want, wcounts = _oracle(mapped, seq_small, KFS, poses, level, flt)
        assert counts.tolist() == wcounts.tolist(), flt
        assert _same_bits(got, want), flt
        # no NaN in the mapped keyframes: there the records must be identical bytes
        n_mapped = int(counts[:2].sum())
        assert got[:n_mapped].tobytes() == want[:n_mapped].tobytes()
        assert counts[0] > 0 and counts[1] > 0
        nan_seen |= bool(np.isnan(got).any())
    if level == 0:
        assert nan_seen                     # the adversarial keyframe reaches the 0 * inf = NaN path


def test_scale_changes_the_filter(mapped):
    flt = mc.FILTERS[4]
    _, c1 = mapped.export_map([4], [mc.POSES[0]], 0, *flt)
    _, c2 = mapped.export_map([4], [mc.POSES[1]], 0, *flt)
    assert c1[0] != c2[0]


def test_many_keyframes_equal_single_exports_and_are_deterministic(mapped):
    # more keyframes than one staging chunk (8), with repeats, in an arbitrary order
    ids = [0, 4, 9, 10, 4, 0, 10, 9, 9, 4, 0, 10, 4, 0, 9, 10, 0, 4, 10]
    poses = [mc.POSES[i % 3] for i in range(len(ids))]
    flt = mc.FILTERS[1]
    got, counts = mapped.export_map(ids, poses, 0, *flt)
    singles = [mapped.export_map([i], [q], 0, *flt) for i, q in zip(ids, poses)]
    assert counts.tolist() == [int(c[0]) for _, c in singles]
    assert got.tobytes() == np.concatenate([p for p, _ in singles]).tobytes()
    again, counts2 = mapped.export_map(ids, poses, 0, *flt)
    assert again.tobytes() == got.tobytes() and counts2.tolist() == counts.tolist()


def _raw(ctx, ids, poses, level, flt, out, capacity, counts, total):
    ids = np.ascontiguousarray(ids, np.int32)
    qts = np.ascontiguousarray(poses, np.float64).reshape(-1, 8)
    f = abi.MapFilter(*flt)
    return ctx.L.lsdgpu_map_export_points(ctx.ptr, ids.size, ids.ctypes.data_as(C.POINTER(C.c_int)),
                                          qts.ctypes.data_as(C.POINTER(C.c_double)), level, C.byref(f),
                                          None if out is None else out.ctypes.data_as(C.c_void_p), capacity,
                                          None if counts is None else counts.ctypes.data_as(C.POINTER(C.c_int)),
                                          None if total is None else C.byref(total))


def test_count_only_and_capacity(mapped):
    ids, poses, flt = KFS, [mc.POSES[0]] * len(KFS), mc.FILTERS[0]
    pts, counts = mapped.export_map(ids, poses, 1, *flt)
    c = np.full(len(ids), -7, np.int32)
    total = C.c_longlong(-1)
    assert _raw(mapped, ids, poses, 1, flt, None, 0, c, total) == 0
    assert c.tolist() == counts.tolist() and total.value == pts.shape[0] == counts.sum()

    # one record short: an error, and neither the guarded buffer nor the counts are touched
    n = pts.shape[0]
    guard = np.full((n + 16, 4), np.float32(-123.5))
    c2 = np.full(len(ids), -7, np.int32)
    t2 = C.c_longlong(-1)
    assert _raw(mapped, ids, poses, 1, flt, guard[8:], n - 1, c2, t2) != 0
    assert (guard == np.float32(-123.5)).all() and (c2 == -7).all() and t2.value == -1
    # exact capacity: the records land inside the guards
    assert _raw(mapped, ids, poses, 1, flt, guard[8:8 + n], n, c2, t2) == 0
    assert guard[8:8 + n].tobytes() == pts.tobytes()
    assert (guard[:8] == np.float32(-123.5)).all() and (guard[8 + n:] == np.float32(-123.5)).all()


def test_rejects_bad_requests(mapped):
    flt, q = mc.FILTERS[0], [mc.POSES[0]]
    for ids, level in (([99], 0), ([11], 0), ([0], -1), ([0], abi.LEVELS)):
        with pytest.raises(abi.LsdGpuError):
            mapped.export_map(ids, q, level, *flt)
    guard = np.full((64, 4), np.float32(7.0))
    assert _raw(mapped, [0, 99], q * 2, 0, flt, guard, 64, None, None) != 0
    assert (guard == 7.0).all()
    pts, counts = mapped.export_map([], np.zeros((0, 8)), 0, *flt)
    assert pts.shape == (0, 4) and counts.size == 0


def test_write_ply_round_trip(mapped, tmp_path):
    pts, _ = mapped.export_map(KFS[:2], [mc.POSES[0], mc.POSES[1]], 0)
    path = tmp_path / "pc.ply"
    abi.write_ply(path, pts)
    data = path.read_bytes()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    header = data[:end].decode("ascii").splitlines()
    assert header == ["ply", "format binary_little_endian 1.0", f"element vertex {pts.shape[0]}", "property float x",
                      "property float y", "property float z", "property float intensity", "end_header"]
    back = np.frombuffer(data[end:], "<f4").reshape(-1, 4)
    assert back.tobytes() == pts.tobytes()
