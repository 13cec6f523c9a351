"""PIN of the oracle: the hand-written C restatement (oracle/lsd_oracle.c) against outputs of the reference's OWN sources
(DepthMap.cpp, SE3Tracker.cpp, Sim3Tracker.cpp, TrackingReference.cpp, Frame.cpp, ... and the vendored Sophus, compiled
unmodified by oracle/ref_build.py) on identical inputs.

* Frame builders, point cloud, stereo constants, and the WHOLE DepthMap (observe / line stereo / fill holes /
  regularise / propagate / createKeyFrame / finalizeKeyFrame) must agree BIT FOR BIT, every field of every pixel.
* Tracking (fp32 sums in another association order on neither side: both are sequential) must agree to fp32
  round-off in every reported quantity, and poses within 1e-5.

Each case below runs one call sequence on one library flavour and returns a record of what it computed.  The records of the
reference-compiled libraries ("ref", "ref_sse") are stored in tests/golden/ref_pin_320x240.json (tests/golden/make_golden.py
writes them where oracle/_ref can be built); the tests run the same cases on the C restatement (False, True) and compare.
Bit-for-bit comparisons of large arrays are made on SHA-256 digests of their bit patterns; values compared with a
tolerance are stored as they are."""
import base64
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from tests.util import IDENT, pose_err

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pin_320x240.json")

FIELDS = ("isValid", "blacklisted", "nextStereoFrameMinID", "validity_counter", "idepth", "idepth_var",
          "idepth_smoothed", "idepth_var_smoothed")


@pytest.fixture(scope="module")
def gold():
    with open(GOLD) as f:
        return json.load(f)


def _bits(a):
    return a.view(np.uint32) if a.dtype == np.float32 else a


def digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(_bits(a).tobytes()).hexdigest()


def pack_mask(m):
    m = np.asarray(m) != 0
    return {"shape": list(m.shape), "bits": base64.b64encode(np.packbits(m.ravel()).tobytes()).decode()}


def unpack_mask(r):
    n = int(np.prod(r["shape"]))
    return np.unpackbits(np.frombuffer(base64.b64decode(r["bits"]), np.uint8))[:n].reshape(r["shape"]).astype(bool)


def hyp_record(h):
    """isValid and blacklisted on every pixel; every other field, as bit patterns, on every valid pixel.  (The reference's
    DepthMapPixelHypothesis() constructor sets only isValid and blacklisted -- DepthMapPixelHypothesis.h:63-64 -- so the
    other fields of a never-valid pixel are uninitialised heap memory in the reference and carry no information.)"""
    va = h["isValid"] != 0
    rec = {"n_valid": int(va.sum()), "isValid": digest(va.astype(np.uint8)), "blacklisted": digest(h["blacklisted"])}
    for f in FIELDS[2:]:
        rec[f] = digest(np.ascontiguousarray(h[f])[va])
    return rec


def assert_hyp_identical(rec, want, what):
    bad = [k for k in want if rec[k] != want[k]]
    assert not bad, f"{what}: {bad} differ (valid pixels: {rec['n_valid']} here, {want['n_valid']} in the reference)"


def _gt_qts(seq, k):
    return np.concatenate([seq.frame_to_ref_qt(k), [1.0]])


class Run:
    """one call sequence on one flavour (False = C restatement, "ref" = reference-compiled); `checks` records the map"""

    def __init__(self, fl, seq, frames, init="gt"):
        self.fl, self.seq, self.frames = fl, seq, frames
        self.checks = {}
        po.set_globals(fl)
        img0, d0 = frames[0]
        self.kf = po.Frame(0, img0, seq.K, fast=fl)
        self.dm = po.DepthMap(seq.w, seq.h, seq.K, fast=fl)
        if init == "gt":
            self.kf.setDepthFromGroundTruth(d0)
            self.dm.initializeFromGTDepth(self.kf)
        else:
            C.CDLL(None).srand(1)               # DepthMap.cpp:898 draws from glibc rand(): same stream on both sides
            self.dm.initializeRandomly(self.kf)
        self.fr = {0: self.kf}

    def add_frame(self, k, qts, itr=0.0, mask=None, parent=0):
        f = po.Frame(k, self.frames[k][0], self.seq.K, fast=self.fl)
        f.set_thisToParent(qts, self.fr[parent])
        f.L.lsdo_frame_set_initialTrackedResidual(f.ptr, float(itr))
        if mask is not None:
            f.refPixelWasGood(create=True)[:] = mask
        self.fr[k] = f

    def check(self, what):
        self.checks[what] = hyp_record(self.dm.current())


def assert_checks_identical(rec, want):
    assert list(rec["checks"]) == list(want["checks"])
    for what in want["checks"]:
        assert_hyp_identical(rec["checks"][what], want["checks"][what], what)


# ------------------------------------------------------------------------------------------------------------
# cases: fl -> record (JSON-serialisable)
# ------------------------------------------------------------------------------------------------------------
def case_frame_builders(fl, seq, frames):
    """Frame.cpp:35-54, 491-630, 643-680, 690-767, 245-293, 775-877"""
    po.set_globals(fl)
    img, d0 = frames[0]
    f = po.Frame(0, img, seq.K, fast=fl)
    f.setDepthFromGroundTruth(d0)
    rec = {}
    for lvl in range(5):
        K, Ki = f.K(lvl)
        rec[f"level{lvl}"] = {"image": digest(f.image(lvl)), "gradients": digest(f.gradients(lvl)), "idepth": digest(f.idepth(lvl)),
                              "idepthVar": digest(f.idepthVar(lvl)), "K": digest(K), "Kinv": digest(Ki)}
    # buildMaxGradients: rows 1 and h-2 read never-written pool memory in the reference (SURVEY App. A-12); interior is defined
    rec["maxGradients_interior"] = digest(f.maxGradients(0)[2:-2])
    rec["numPoints"] = int(f.L.lsdo_frame_numPoints(f.ptr))
    rec["meanIdepth"] = float(np.float32(f.L.lsdo_frame_meanIdepth(f.ptr)))
    return rec


def case_point_cloud(fl, seq, frames):
    """TrackingReference::makePointCloud (TrackingReference.cpp:96-147)"""
    po.set_globals(fl)
    img, d0 = frames[0]
    f = po.Frame(0, img, seq.K, fast=fl)
    f.setDepthFromGroundTruth(d0)
    rec = {}
    for lvl in (1, 2, 3, 4):
        pc = f.point_cloud(lvl)
        rec[f"level{lvl}"] = {"n": len(pc[0]), "arrays": [digest(x) for x in pc]}
    return rec


def case_prepare_for_stereo(fl, seq, frames):
    """Frame::prepareForStereoWith (Frame.cpp:295-317): Sim3 inverse, K*R*s, columns of thisToOther_R"""
    po.set_globals(fl)
    rng = np.random.default_rng(5)
    K = np.ascontiguousarray(seq.K, np.float32).reshape(9)
    fp, dp = C.POINTER(C.c_float), C.POINTER(C.c_double)
    out = []
    for trial in range(8):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        qts = np.concatenate([q, rng.normal(size=3) * 0.3, [np.exp(rng.normal() * 0.2) if trial else 1.0]])
        kf = po.Frame(0, frames[0][0], seq.K, fast=fl)
        f = po.Frame(3, frames[3][0], seq.K, fast=fl)
        o = np.zeros(30, np.float32)
        f.L.lsdo_ref_prepareForStereoWith(f.ptr, kf.ptr, qts.ctypes.data_as(dp), K.ctypes.data_as(fp), o.ctypes.data_as(fp))
        out.append([int(x) for x in o.view(np.uint32)])
    return {"bits": out}


def case_depthmap_update_sequence(fl, seq, frames):
    """updateKeyframe x6 (1, 2 and 3 reference frames, with and without the tracking mask) -- DepthMap.cpp:111-473,
    1072-1213, 1442-1972, 656-880 and Frame::setDepth, every field of every pixel"""
    t = Run(fl, seq, frames, "gt")
    rng = np.random.default_rng(11)
    w1, h1 = seq.w // 2, seq.h // 2
    groups = [[1], [2, 3], [4], [5, 6, 7], [8], [9]]
    kf_depth = {}
    for gi, ks in enumerate(groups):
        for k in ks:
            mask = (rng.random((h1, w1)) > 0.15).astype(np.uint8) if gi % 2 == 0 else None
            t.add_frame(k, _gt_qts(seq, k), itr=0.05 * gi, mask=mask)
        t.dm.updateKeyframe([t.fr[k] for k in ks])
        t.check(f"updateKeyframe {ks}")
        # the keyframe's exported depth (Frame::setDepth + pyramids) as the tracker will read it
        kf_depth[f"updateKeyframe {ks}"] = [[digest(t.kf.idepth(lvl)), digest(t.kf.idepthVar(lvl))] for lvl in range(5)]
    return {"checks": t.checks, "kf_depth": kf_depth}


def case_depthmap_random_init(fl, seq, frames):
    """random hypotheses drive doLineStereo / observeDepthUpdate through their failure, inconsistency and skip branches"""
    t = Run(fl, seq, frames, "random")
    t.check("initializeRandomly")
    for k in (4, 6, 8, 10, 12):
        t.add_frame(k, _gt_qts(seq, k))
        t.dm.updateKeyframe([t.fr[k]])
        t.check(f"random-init updateKeyframe [{k}]")
    return {"checks": t.checks}


def case_depthmap_individual_passes(fl, seq, frames):
    """observeDepth, regularizeDepthMapFillHoles, regularizeDepthMap<true/false> one by one (private members of the
    reference class called as they are)"""
    t = Run(fl, seq, frames, "gt")
    t.add_frame(2, _gt_qts(seq, 2))
    t.add_frame(3, _gt_qts(seq, 3))
    t.dm.observeDepth([t.fr[2], t.fr[3]])
    t.check("observeDepth")
    t.dm.regularizeFillHoles()
    t.check("fillHoles")
    t.dm.regularize(False, 24)
    t.check("regularize<false>")
    t.dm.regularize(True, 24)
    t.check("regularize<true>")
    return {"checks": t.checks, "integral": digest(t.dm.integral())}


def case_create_keyframe_and_finalize(fl, seq, frames):
    """finalizeKeyFrame + createKeyFrame (propagateDepth with the tracking mask, 2x regularise, fill holes, rescale,
    pose scale) -- DepthMap.cpp:475-653, 1222-1327, 1363-1395; then mapping continues on the new keyframe, including with
    frames that were tracked on the PREVIOUS keyframe (:1085-1099).
    The scene is rescaled so that keyframe 0 already has mean inverse depth 1, as every keyframe after the first has in a real
    run: doLineStereo only accepts a reference frame whose depth ratio to the keyframe is within 0.7..1.4 (:119 `rescaleFactor`),
    so with a 2x scale jump between keyframes the off-parent frames would be rejected pixel by pixel and test nothing."""
    d0 = frames[0][1]
    sc = float(np.mean(1.0 / d0[d0 > 0]))
    frames = {k: (frames[k][0], (frames[k][1] * sc).astype(np.float32)) for k in range(13)}

    def qts(k, ref=0):
        q = seq.frame_to_ref_qt(k, ref=ref).copy()
        q[4:7] *= sc
        return np.concatenate([q, [1.0]])
    t = Run(fl, seq, frames, "gt")
    rng = np.random.default_rng(3)
    w1, h1 = seq.w // 2, seq.h // 2
    for k in (1, 2, 3):
        t.add_frame(k, qts(k), itr=0.1)
        t.dm.updateKeyframe([t.fr[k]])
    t.check("before finalize")
    t.dm.finalizeKeyFrame()
    t.check("finalizeKeyFrame")
    mask = (rng.random((h1, w1)) > 0.1).astype(np.uint8)
    t.add_frame(9, qts(9), itr=0.1, mask=mask)
    t.dm.createKeyFrame(t.fr[9])
    t.check("createKeyFrame")
    pa = t.fr[9].thisToParent()                                   # rescaled Sim3 (DepthMap.cpp:1305)
    # frames tracked on the PREVIOUS keyframe, mapped on the new one: refToKf comes from the chained absolute poses (:1099), and the
    # tracking-mask gate of :245 / :322 is off for them
    for k in (4, 5):
        t.add_frame(k, qts(k), itr=0.07, mask=mask, parent=0)
    before = t.dm.current().copy()
    t.dm.updateKeyframe([t.fr[4], t.fr[5]])
    t.check("updateKeyframe with frames tracked on the previous keyframe")
    after = t.dm.current()
    both = (before["isValid"] != 0) & (after["isValid"] != 0)
    observed = int((before["idepth"][both] != after["idepth"][both]).sum())
    # frames tracked on the NEW keyframe
    for k in (10, 11):
        q = qts(k, ref=9)
        q[4:7] /= pa[7]                                           # the new keyframe's units
        t.add_frame(k, q, itr=0.1, parent=9)
        t.dm.updateKeyframe([t.fr[k]])
        t.check(f"updateKeyframe on new keyframe [{k}]")
    q = qts(12, ref=9)
    q[4:7] /= pa[7]
    t.add_frame(12, q, itr=0.1, parent=9)
    t.add_frame(6, qts(6), itr=0.05, mask=mask, parent=0)
    t.dm.updateKeyframe([t.fr[6], t.fr[12]])                      # mixed parents in one call
    t.check("updateKeyframe with mixed tracking parents")
    return {"checks": t.checks, "new_kf_thisToParent": [float(x) for x in pa], "observed_after_change": observed}


def case_se3_single_evaluation(fl, seq, frames):
    """calcResidualAndBuffers + calcWeightsAndResidual + calculateWarpUpdate (SE3Tracker.cpp:885-1029, 749-790,
    1258-1299, LGSX.h:184-402), the reference's private members called directly"""
    po.set_globals(fl)
    kf = po.Frame(0, frames[0][0], seq.K, fast=fl)
    kf.setDepthFromGroundTruth(frames[0][1])
    f = po.Frame(3, frames[3][0], seq.K, fast=fl)
    inv = np.zeros(7)
    g = np.ascontiguousarray(seq.frame_to_ref_qt(3), np.float64)
    po.lib(False).lsdo_se3d_inverse(g.ctypes.data_as(C.POINTER(C.c_double)), inv.ctypes.data_as(C.POINTER(C.c_double)))
    pose = inv.astype(np.float32)
    rec = {}
    for lvl in (4, 3, 2, 1):
        r = po.se3_eval(kf, f, lvl, pose, 1.0, 0.0, po.default_track_settings(fl), write_mask=(lvl == 1))
        rec[f"level{lvl}"] = {k: float(getattr(r, k)) for k in ("warpedSize", "goodCount", "badCount", "pointUsage", "meanUnweightedRes",
                                                                 "meanWeightedRes", "lsError", "meanRes", "affine_a_lastIt", "affine_b_lastIt")}
        rec[f"level{lvl}"]["A"] = [float(x) for x in r.A]
        rec[f"level{lvl}"]["b"] = [float(x) for x in r.b]
    rec["mask"] = pack_mask(f.refPixelWasGood(create=False))
    return rec


def case_se3_track(fl, seq, frames):
    """SE3Tracker::trackFrame over a tracked + mapped sequence: pose, every reported statistic, the good-mask"""
    po.set_globals(fl, useSSE=1) if fl is True else po.set_globals(fl)
    kf = po.Frame(0, frames[0][0], seq.K, fast=fl)
    kf.setDepthFromGroundTruth(frames[0][1])
    dm = po.DepthMap(seq.w, seq.h, seq.K, fast=fl)
    dm.initializeFromGTDepth(kf)
    st = po.default_track_settings(fl)
    last, out, keep = IDENT, [], []
    for k in range(1, 7):
        f = po.Frame(k, frames[k][0], seq.K, fast=fl)
        keep.append(f)
        kf.L.lsdo_frame_set_depthHasBeenUpdatedFlag(kf.ptr, 0)
        r = po.se3_track(kf, f, last, st)
        last = np.array(r.frameToRef_qt)
        out.append({"pose": [float(x) for x in last],
                    "stats": [float(x) for x in (r.lastResidual, r.pointUsage, r.lastGoodCount, r.lastBadCount, r.lastMeanRes,
                                                 r.affineEstimation_a, r.affineEstimation_b, r.diverged, r.trackingWasGood,
                                                 r.initialTrackedResidual)],
                    "mask": pack_mask(f.refPixelWasGood(create=False))})
        dm.updateKeyframe([f])
    return out


def case_track_frame3_from_identity(fl, seq, frames):
    po.set_globals(fl, useSSE=1) if fl is True else po.set_globals(fl)
    kf = po.Frame(0, frames[0][0], seq.K, fast=fl)
    kf.setDepthFromGroundTruth(frames[0][1])
    f = po.Frame(3, frames[3][0], seq.K, fast=fl)
    return [float(x) for x in po.se3_track(kf, f, IDENT, po.default_track_settings(fl)).frameToRef_qt]


def case_bench_loop(fl, seq, frames):
    """the loop bench.py and the full-size GPU tests run (oracle/cpu_stream.py: track, map, forced finalizeKeyFrame +
    createKeyFrame every 10 frames)"""
    from oracle.cpu_stream import CpuStream
    po.set_globals(fl)
    cs = CpuStream(seq, fl, kf_every=10)
    cs.init_gt(0, *frames[0])
    for k in range(1, 26):
        cs.step(k, frames[k][0])
    return {"poses": np.array(cs.poses).tolist(), "kf_changes": list(cs.kf_changes), "map": hyp_record(cs.dm.current())}


# reference-compiled records: case name -> {flavour: record}
CASES = {"frame_builders": (case_frame_builders, ("ref",)), "point_cloud": (case_point_cloud, ("ref",)),
         "prepare_for_stereo": (case_prepare_for_stereo, ("ref",)),
         "depthmap_update_sequence": (case_depthmap_update_sequence, ("ref",)),
         "depthmap_random_init": (case_depthmap_random_init, ("ref",)),
         "depthmap_individual_passes": (case_depthmap_individual_passes, ("ref",)),
         "create_keyframe_and_finalize": (case_create_keyframe_and_finalize, ("ref",)),
         "se3_single_evaluation": (case_se3_single_evaluation, ("ref",)),
         "se3_track": (case_se3_track, ("ref", "ref_sse")),
         "track_frame3_from_identity": (case_track_frame3_from_identity, ("ref", "ref_sse")),
         "bench_loop": (case_bench_loop, ("ref",))}


def reference_records(seq, frames):
    return {name: {fl: fn(fl, seq, frames) for fl in fls} for name, (fn, fls) in CASES.items()}


# ------------------------------------------------------------------------------------------------------------
# tests: the C restatement against the stored reference records
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(not po.ref_available(), reason="the reference sources are not present to build oracle/_ref")
def test_vendored_sophus_suite_passes_on_the_shim():
    """thirdparty/Sophus/sophus/test_{so3,se3,sim3,rxso3}.cpp, compiled unmodified against oracle/ref_shim/Eigen"""
    import subprocess
    from oracle import ref_build
    ref_build.build()
    for t in ref_build.SOPHUS_TESTS:
        r = subprocess.run([os.path.join(ref_build.OUT, f"test_{t}")], capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stderr[-500:]
        assert "passed" in r.stderr and "failed" not in r.stderr


def test_frame_builders_bit_exact(seq_small, frames_small, gold):
    rec, want = case_frame_builders(False, seq_small, frames_small), gold["frame_builders"]["ref"]
    for lvl in range(5):
        for k, v in want[f"level{lvl}"].items():
            assert rec[f"level{lvl}"][k] == v, (lvl, k)
    assert rec["maxGradients_interior"] == want["maxGradients_interior"]
    assert rec["numPoints"] == want["numPoints"]
    assert rec["meanIdepth"] == want["meanIdepth"]


def test_point_cloud_bit_exact(seq_small, frames_small, gold):
    rec, want = case_point_cloud(False, seq_small, frames_small), gold["point_cloud"]["ref"]
    for lvl in (1, 2, 3, 4):
        a, b = rec[f"level{lvl}"], want[f"level{lvl}"]
        assert a["n"] == b["n"] > 100, lvl
        assert a["arrays"] == b["arrays"], lvl


def test_prepare_for_stereo_bit_exact(seq_small, frames_small, gold):
    rec, want = case_prepare_for_stereo(False, seq_small, frames_small), gold["prepare_for_stereo"]["ref"]
    for trial, (a, b) in enumerate(zip(rec["bits"], want["bits"], strict=True)):
        a, b = np.array(a, np.uint32), np.array(b, np.uint32)
        assert np.array_equal(a, b), (trial, a.view(np.float32) - b.view(np.float32))


def test_depthmap_update_sequence_bit_exact(seq_small, frames_small, gold):
    rec, want = case_depthmap_update_sequence(False, seq_small, frames_small), gold["depthmap_update_sequence"]["ref"]
    assert_checks_identical(rec, want)
    assert rec["kf_depth"] == want["kf_depth"]
    assert list(rec["checks"].values())[-1]["n_valid"] > 15000


def test_depthmap_random_init_every_branch_bit_exact(seq_small, frames_small, gold):
    rec, want = case_depthmap_random_init(False, seq_small, frames_small), gold["depthmap_random_init"]["ref"]
    assert_checks_identical(rec, want)
    assert list(rec["checks"].values())[-1]["n_valid"] > 5000


def test_depthmap_individual_passes_bit_exact(seq_small, frames_small, gold):
    rec, want = case_depthmap_individual_passes(False, seq_small, frames_small), gold["depthmap_individual_passes"]["ref"]
    assert_checks_identical(rec, want)
    assert rec["integral"] == want["integral"]


def test_create_keyframe_and_finalize_bit_exact(seq_small, frames_small, gold):
    rec, want = case_create_keyframe_and_finalize(False, seq_small, frames_small), gold["create_keyframe_and_finalize"]["ref"]
    assert_checks_identical(rec, want)
    pa, pb = np.array(rec["new_kf_thisToParent"]), np.array(want["new_kf_thisToParent"])
    assert np.allclose(pa, pb, rtol=0, atol=1e-12), pa - pb
    assert 0.8 < pa[7] < 1.25
    n = rec["checks"]["updateKeyframe with frames tracked on the previous keyframe"]["n_valid"]
    assert n > 10000 and rec["observed_after_change"] > 2000                 # they did observe


def test_se3_single_evaluation_matches_reference_compiled(seq_small, frames_small, gold):
    rec, want = case_se3_single_evaluation(False, seq_small, frames_small), gold["se3_single_evaluation"]["ref"]
    for lvl in (4, 3, 2, 1):
        ra, rb = rec[f"level{lvl}"], want[f"level{lvl}"]
        assert ra["warpedSize"] == rb["warpedSize"] > 50
        assert (ra["goodCount"], ra["badCount"]) == (rb["goodCount"], rb["badCount"])
        assert ra["pointUsage"] == rb["pointUsage"]
        for f in ("meanUnweightedRes", "meanWeightedRes", "lsError", "meanRes", "affine_a_lastIt", "affine_b_lastIt"):
            x, y = ra[f], rb[f]
            assert abs(x - y) <= 2e-6 * max(abs(y), 1.0), (lvl, f, x, y)
        A, B = np.array(ra["A"]), np.array(rb["A"])
        assert np.abs(A - B).max() <= 2e-6 * np.abs(B).max(), lvl
        assert np.abs(np.array(ra["b"]) - np.array(rb["b"])).max() <= 2e-6 * np.abs(np.array(rb["b"])).max() + 1e-9, lvl
    assert np.array_equal(unpack_mask(rec["mask"]), unpack_mask(want["mask"]))


@pytest.mark.parametrize("pair", [(False, "ref"), (True, "ref_sse")], ids=["scalar", "sse"])
def test_se3_track_matches_reference_compiled(seq_small, frames_small, gold, pair):
    """'sse' compares the oracle's restatement of the SSE loops (SE3Tracker.cpp:492-575, 1033-1130, LGSX.h:205-386) with the
    stock ENABLE_SSE build of the reference."""
    fa, fb = pair
    rec, want = case_se3_track(fa, seq_small, frames_small), gold["se3_track"][fb]
    assert len(rec) == len(want)
    for k, (x, y) in enumerate(zip(rec, want)):
        ma, mb = unpack_mask(x["mask"]), unpack_mask(y["mask"])
        if fa is False:
            # scalar path, strict IEEE on both sides: the restatement reproduces the reference-compiled tracker BIT FOR BIT
            # (pose as doubles, every statistic, the mask) -- same sequential sums, same LDLT, same Sophus arithmetic
            assert np.array_equal(x["pose"], y["pose"]), (k, np.subtract(x["pose"], y["pose"]))
            for i, (a, b) in enumerate(zip(x["stats"], y["stats"])):
                assert np.float32(a) == np.float32(b), (k, i, a, b)
            assert np.array_equal(ma, mb)
            continue
        # timing flavours: both are -O3 builds with FMA contraction left to the compiler, so only fp32 round-off agreement
        dt, ang = pose_err(x["pose"], y["pose"])
        assert dt <= 1e-4 and ang <= 1e-6, (k, dt, ang)
        xs, ys = x["stats"], y["stats"]             # lastResidual, pointUsage, good, bad, meanRes, affine a, b, diverged, good, itr
        for i in (0, 1, 5, 9):
            assert abs(xs[i] - ys[i]) <= 2e-4 * max(abs(ys[i]), 1.0), (k, i, xs[i], ys[i])
        assert abs(xs[4] - ys[4]) <= 1e-2 and abs(xs[6] - ys[6]) <= 1e-2    # mean signed residual, affine b (grey levels): fp32 cancellation
        assert abs(xs[2] - ys[2]) <= 3 and abs(xs[3] - ys[3]) <= 3, (k, xs[2:4], ys[2:4])       # good / bad counts
        assert xs[7] == ys[7] and xs[8] == ys[8]
        assert (ma != mb).mean() <= 1e-3


def test_sse_vs_scalar_gap_of_the_reference_itself(seq_small, frames_small, gold):
    """The stock build defines ENABLE_SSE (CMakeLists.txt:37-43): _mm_rcp_ps weights, N mod 4 points dropped.  This
    MEASURES how far the reference's two code paths are apart on the same input (documented in DESIGN.md section 2):
    the scalar path is the parity target of the CUDA kernels, the SSE path the timing baseline."""
    out = gold["track_frame3_from_identity"]
    # the stored scalar pose is the one the restatement computes, bit for bit
    assert case_track_frame3_from_identity(False, seq_small, frames_small) == out["ref"]
    dt, ang = pose_err(out["ref_sse"], out["ref"])
    gt = seq_small.frame_to_ref_qt(3)
    e_scalar, _ = pose_err(out["ref"], gt)
    e_sse, _ = pose_err(out["ref_sse"], gt)
    print(f"reference SSE vs reference scalar: translation {dt:.2e} rel, rotation {ang:.2e} rad; "
          f"vs ground truth: scalar {e_scalar:.2e}, SSE {e_sse:.2e}")
    assert 1e-4 < dt < 5e-2             # both minimise the same cost; they are NOT within 1e-4 of each other
    assert abs(e_scalar - e_sse) < 2e-2 # and neither is closer to the ground truth than the other by more than that


def test_bench_loop_with_keyframe_changes_bit_exact(seq_small, frames_small, gold):
    """C oracle vs reference-compiled: every pose equal as doubles, final map identical"""
    rec, want = case_bench_loop(False, seq_small, frames_small), gold["bench_loop"]["ref"]
    assert rec["kf_changes"] == want["kf_changes"] == [10, 20]
    assert np.array_equal(rec["poses"], want["poses"])
    assert_hyp_identical(rec["map"], want["map"], "after 25 frames and 2 keyframe changes")
