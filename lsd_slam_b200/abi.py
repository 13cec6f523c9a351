"""ctypes binding of the C ABI (include/lsdgpu.h -> liblsdgpu.so) plus thin Python mirrors of the reference's
public interface for the hot path (``SE3Tracker.trackFrame``, ``DepthMap.updateKeyframe`` /
``createKeyFrame`` -- Tracking/SE3Tracker.h:65-68, DepthEstimation/DepthMap.h:58,63).

This is the product path: it loads the CUDA library and nothing else.  There is NO CPU fallback -- a missing
or unloadable ``liblsdgpu.so`` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblsdgpu.so")
LEVELS = 5

EVAL_NSUMS = 40
ALLREDUCE_FN = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(C.c_float), C.c_int)

BUF_IMAGE, BUF_GRADIENTS, BUF_MAXGRAD, BUF_IDEPTH, BUF_IDEPTH_VAR, BUF_GOODMASK = range(6)


class Hyp(C.Structure):
    _fields_ = [("isValid", C.c_uint8), ("_pad", C.c_uint8 * 3), ("blacklisted", C.c_int32),
                ("nextStereoFrameMinID", C.c_float), ("validity_counter", C.c_int32),
                ("idepth", C.c_float), ("idepth_var", C.c_float),
                ("idepth_smoothed", C.c_float), ("idepth_var_smoothed", C.c_float)]


HYP_DTYPE = np.dtype([("isValid", np.uint8), ("_pad", np.uint8, 3), ("blacklisted", np.int32),
                      ("nextStereoFrameMinID", np.float32), ("validity_counter", np.int32),
                      ("idepth", np.float32), ("idepth_var", np.float32),
                      ("idepth_smoothed", np.float32), ("idepth_var_smoothed", np.float32)])


POINT_DENSE = np.dtype([("idepth", np.float32), ("idepth_var", np.float32), ("color", np.uint8, (4,))])     # InputPointDense


class RefDesc(C.Structure):
    """lsdgpu_ref_desc (include/lsdgpu.h)"""
    _fields_ = [("frame_id", C.c_int32), ("tracked_on_kf", C.c_int32), ("refToKf_qts", C.c_double * 8)]


class Globals(C.Structure):
    _fields_ = [("minUseGrad", C.c_float), ("cameraPixelNoise2", C.c_float), ("depthSmoothingFactor", C.c_float),
                ("allowNegativeIdepths", C.c_int), ("useSubpixelStereo", C.c_int),
                ("useAffineLightningEstimation", C.c_int)]


class TrackSettings(C.Structure):
    _fields_ = [("lambdaSuccessFac", C.c_float), ("lambdaFailFac", C.c_float),
                ("lambdaInitial", C.c_float * LEVELS), ("stepSizeMin", C.c_float * LEVELS),
                ("convergenceEps", C.c_float * LEVELS), ("maxItsPerLvl", C.c_int * LEVELS),
                ("huber_d", C.c_float), ("var_weight", C.c_float)]


class TrackResult(C.Structure):
    _fields_ = [("frameToRef_qt", C.c_double * 7),
                ("pointUsage", C.c_float), ("lastGoodCount", C.c_float), ("lastBadCount", C.c_float),
                ("lastMeanRes", C.c_float), ("lastResidual", C.c_float),
                ("affineEstimation_a", C.c_float), ("affineEstimation_b", C.c_float),
                ("diverged", C.c_int), ("trackingWasGood", C.c_int),
                ("numCalcResidualCalls", C.c_int * LEVELS), ("numCalcWarpUpdateCalls", C.c_int * LEVELS),
                ("initialTrackedResidual", C.c_float)]


class EvalResult(C.Structure):
    _fields_ = [("A", C.c_float * 36), ("b", C.c_float * 6), ("lsError", C.c_float),
                ("meanWeightedRes", C.c_float), ("meanUnweightedRes", C.c_float), ("warpedSize", C.c_int),
                ("pointUsage", C.c_float), ("goodCount", C.c_float), ("badCount", C.c_float), ("meanRes", C.c_float),
                ("affine_a_lastIt", C.c_float), ("affine_b_lastIt", C.c_float),
                ("sxx", C.c_float), ("syy", C.c_float), ("sx", C.c_float), ("sy", C.c_float), ("sw", C.c_float)]


# every symbol include/lsdgpu.h declares: (name, restype, argtypes)
_vp, _fp, _dp, _ip, _u8p = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_uint8)
class Sim3Result(C.Structure):
    _fields_ = [("frameToRef_qts", C.c_double * 8), ("lastSim3Hessian", C.c_float * 49),
                ("lastResidual", C.c_float), ("lastDepthResidual", C.c_float), ("lastPhotometricResidual", C.c_float),
                ("pointUsage", C.c_float), ("affineEstimation_a", C.c_float), ("affineEstimation_b", C.c_float),
                ("diverged", C.c_int),
                ("numCalcResidualCalls", C.c_int * LEVELS), ("numCalcWarpUpdateCalls", C.c_int * LEVELS)]


class Sim3EvalResult(C.Structure):
    _fields_ = [("A", C.c_float * 49), ("b", C.c_float * 7), ("num_constraints", C.c_int),
                ("sumResD", C.c_float), ("sumResP", C.c_float), ("numTermsD", C.c_int), ("numTermsP", C.c_int),
                ("mean", C.c_float), ("meanD", C.c_float), ("meanP", C.c_float), ("warpedSize", C.c_int),
                ("pointUsage", C.c_float), ("affine_a_lastIt", C.c_float), ("affine_b_lastIt", C.c_float)]


class MapFilter(C.Structure):
    """lsdgpu_map_filter: the point filter of lsd_slam_viewer's KeyFrameDisplay::flushPC (KeyFrameDisplay.cpp:274-307)"""
    _fields_ = [("scaledDepthVarTH", C.c_float), ("absDepthVarTH", C.c_float), ("minNearSupport", C.c_int)]


def write_ply(path, points: np.ndarray) -> None:
    """Write (N, 4) float32 map points (x, y, z, intensity) as the binary PLY of lsd_slam_viewer's KeyFrameGraphDisplay::draw
    (header KeyFrameGraphDisplay.cpp:75-82, records KeyFrameDisplay.cpp:328-333).  The viewer's copy loop (:85) also appends one
    stray 0xFF byte after the last record (it writes the EOF of f3.get()); that byte is not written here."""
    pts = np.ascontiguousarray(points, np.float32).reshape(-1, 4)
    header = ("ply\n"
              "format binary_little_endian 1.0\n"
              f"element vertex {pts.shape[0]}\n"
              "property float x\n"
              "property float y\n"
              "property float z\n"
              "property float intensity\n"
              "end_header\n")
    with open(path, "wb") as f:
        f.write(header.encode("ascii"))
        f.write(pts.astype("<f4", copy=False).tobytes())


SYMBOLS = [
    ("lsdgpu_create", C.c_int, [C.c_int, C.c_int, C.c_int, _fp, C.c_int, C.POINTER(_vp)]),
    ("lsdgpu_destroy", None, [_vp]),
    ("lsdgpu_last_error", C.c_char_p, [_vp]),
    ("lsdgpu_abi_version", C.c_int, []),
    ("lsdgpu_set_globals", C.c_int, [_vp, C.POINTER(Globals)]),
    ("lsdgpu_get_globals", C.c_int, [_vp, C.POINTER(Globals)]),
    ("lsdgpu_default_globals", None, [C.POINTER(Globals)]),
    ("lsdgpu_default_track_settings", None, [C.POINTER(TrackSettings)]),
    ("lsdgpu_synchronize", C.c_int, [_vp]),
    ("lsdgpu_launch_count", C.c_longlong, [_vp]),
    ("lsdgpu_timer_begin", C.c_int, [_vp, C.c_int]),
    ("lsdgpu_timer_end", C.c_int, [_vp, C.c_int]),
    ("lsdgpu_timer_elapsed_ms", C.c_int, [_vp, C.c_int, _fp]),
    ("lsdgpu_track_kernel_stats", C.c_int, [_vp, C.c_int, _dp, C.POINTER(C.c_longlong), _dp]),
    ("lsdgpu_frame_upload_u8", C.c_int, [_vp, C.c_int, _u8p]),
    ("lsdgpu_frame_release", C.c_int, [_vp, C.c_int]),
    ("lsdgpu_stage_reserve", C.c_int, [_vp, C.c_int]),
    ("lsdgpu_stage_put", C.c_int, [_vp, C.c_int, _u8p]),
    ("lsdgpu_frame_from_stage", C.c_int, [_vp, C.c_int, C.c_int]),
    ("lsdgpu_frame_download", C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp]),
    ("lsdgpu_frame_set_depth_gt", C.c_int, [_vp, C.c_int, _fp, C.c_float]),
    ("lsdgpu_frame_set_idepth", C.c_int, [_vp, C.c_int, _fp, _fp]),
    ("lsdgpu_frame_set_pose", C.c_int, [_vp, C.c_int, _dp, C.c_int, C.c_float]),
    ("lsdgpu_frame_get_pose", C.c_int, [_vp, C.c_int, _dp, _ip, _fp]),
    ("lsdgpu_frame_get_counters", C.c_int, [_vp, C.c_int, _ip, _ip]),
    ("lsdgpu_frame_set_counters", C.c_int, [_vp, C.c_int, C.c_int, C.c_int]),
    ("lsdgpu_frame_get_depth_stats", C.c_int, [_vp, C.c_int, _fp, _ip, _ip]),
    ("lsdgpu_frame_clear_good_mask", C.c_int, [_vp, C.c_int]),
    ("lsdgpu_ref_import", C.c_int, [_vp, C.c_int]),
    ("lsdgpu_se3_eval", C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _fp, C.c_float, C.c_float, C.POINTER(TrackSettings), C.c_int, C.POINTER(EvalResult)]),
    ("lsdgpu_se3_track", C.c_int, [_vp, C.c_int, C.c_int, _dp, C.POINTER(TrackSettings), C.c_int, C.POINTER(TrackResult)]),
    ("lsdgpu_track_and_map", C.c_int, [_vp, C.c_int, C.c_int, _u8p, C.c_int, _dp, C.POINTER(TrackSettings), C.c_int, C.c_int, C.POINTER(TrackResult), _dp]),
    ("lsdgpu_undistorter_ptam_prepare", C.c_int, [_fp, C.c_int, C.c_int, _fp, C.c_int, C.c_int, _fp, _fp, _fp]),
    ("lsdgpu_undistorter_validate_tables", C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _fp, _fp]),
    ("lsdgpu_set_undistorter", C.c_int, [_vp, C.c_int, C.c_int, _fp, _fp]),
    ("lsdgpu_undistort_u8", C.c_int, [_vp, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]),
    ("lsdgpu_frame_upload_distorted_u8", C.c_int, [_vp, C.c_int, C.POINTER(C.c_uint8)]),
    ("lsdgpu_keyframe_pack_pointcloud", C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    ("lsdgpu_map_export_points", C.c_int, [_vp, C.c_int, _ip, _dp, C.c_int, C.POINTER(MapFilter), _vp, C.c_longlong, _ip,
                                           C.POINTER(C.c_longlong)]),
    ("lsdgpu_frame_take_reactivation_data", C.c_int, [_vp, C.c_int]),
    ("lsdgpu_frame_download_reactivation_data", C.c_int, [_vp, C.c_int, _fp, _fp, C.POINTER(C.c_uint8)]),
    ("lsdgpu_depth_set_from_existing_kf", C.c_int, [_vp, C.c_int]),
    ("lsdgpu_sim3_eval", C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _dp, C.c_float, C.c_float, C.POINTER(TrackSettings), C.POINTER(Sim3EvalResult)]),
    ("lsdgpu_sim3_track", C.c_int, [_vp, C.c_int, C.c_int, _dp, C.c_int, C.c_int, C.POINTER(TrackSettings), C.POINTER(Sim3Result)]),
    ("lsdgpu_sim3_track_batch", C.c_int, [_vp, C.c_int, _ip, _ip, _dp, C.c_int, C.c_int, C.POINTER(TrackSettings), C.POINTER(Sim3Result)]),
    ("lsdgpu_frame_set_perma_ref", C.c_int, [_vp, C.c_int, _ip]),
    ("lsdgpu_perma_overlap_batch", C.c_int, [_vp, C.c_int, _ip, _dp, _fp]),
    ("lsdgpu_perma_track_batch", C.c_int, [_vp, C.c_int, _ip, C.c_int, _dp, C.POINTER(TrackResult)]),
    ("lsdgpu_se3_track_sharded", C.c_int, [_vp, C.c_int, C.c_int, _dp, C.POINTER(TrackSettings), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(TrackResult)]),
    ("lsdgpu_depth_reset", C.c_int, [_vp]),
    ("lsdgpu_depth_is_valid", C.c_int, [_vp]),
    ("lsdgpu_depth_invalidate", C.c_int, [_vp]),
    ("lsdgpu_depth_init_from_gt", C.c_int, [_vp, C.c_int]),
    ("lsdgpu_depth_set_hypotheses", C.c_int, [_vp, C.c_int, C.POINTER(Hyp), C.c_int, C.c_int]),
    ("lsdgpu_depth_update_keyframe", C.c_int, [_vp, _ip, C.c_int]),
    ("lsdgpu_depth_update_keyframe_refs", C.c_int, [_vp, C.c_void_p, C.c_int]),
    ("lsdgpu_peer_export", C.c_int, [_vp, C.c_void_p]),
    ("lsdgpu_peer_attach", C.c_int, [_vp, C.c_int, C.c_int, C.c_void_p]),
    ("lsdgpu_peer_detach", C.c_int, [_vp]),
    ("lsdgpu_depth_create_keyframe", C.c_int, [_vp, C.c_int, _dp]),
    ("lsdgpu_seq_sum_f32", C.c_int, [_vp, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    ("lsdgpu_depth_finalize_keyframe", C.c_int, [_vp]),
    ("lsdgpu_depth_active_keyframe", C.c_int, [_vp]),
    ("lsdgpu_depth_download", C.c_int, [_vp, C.POINTER(Hyp)]),
    ("lsdgpu_depth_download_integral", C.c_int, [_vp, C.POINTER(C.c_int32)]),
    ("lsdgpu_depth_observe", C.c_int, [_vp, _ip, C.c_int]),
    ("lsdgpu_depth_regularize_fill_holes", C.c_int, [_vp]),
    ("lsdgpu_depth_regularize", C.c_int, [_vp, C.c_int, C.c_int]),
    ("lsdgpu_depth_propagate", C.c_int, [_vp, C.c_int]),
]

_lib = None


def load():
    """Load liblsdgpu.so (loudly: raises if the extension is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    global LIB_PATH
    if os.environ.get("LSDGPU_LIB"):                 # A/B runs of two builds of the library (scripts/ab_track.py, profiling)
        LIB_PATH = os.path.abspath(os.environ["LSDGPU_LIB"])
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} not found: build it with `python -m lsd_slam_b200.build` "
                           "(the product path has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args
    _lib = L
    return L


class LsdGpuError(RuntimeError):
    pass


class UndistorterPTAM:
    """Mirror of lsd_slam::UndistorterPTAM (util/Undistorter.h:96-160) with the calibration file's lines already parsed.
    out_calib: "crop", "full" or (fx, fy, cx, cy, 0).  Host-only; `install(ctx)` puts the tables on the device."""

    def __init__(self, in_calib, in_size, out_calib, out_size):
        self.in_w, self.in_h = in_size
        self.out_w, self.out_h = out_size
        ic = np.ascontiguousarray(in_calib, np.float32)
        oc = np.zeros(5, np.float32)
        if isinstance(out_calib, str):
            oc[0] = {"crop": -1, "full": -2}[out_calib]
        else:
            oc[:] = out_calib
        self.remapX = np.zeros((self.out_h, self.out_w), np.float32)
        self.remapY = np.zeros((self.out_h, self.out_w), np.float32)
        K = np.zeros(9, np.float32)
        self.status = load().lsdgpu_undistorter_ptam_prepare(ic.ctypes.data_as(_fp), self.in_w, self.in_h, oc.ctypes.data_as(_fp),
                                                             self.out_w, self.out_h, self.remapX.ctypes.data_as(_fp),
                                                             self.remapY.ctypes.data_as(_fp), K.ctypes.data_as(_fp))
        if self.status < 0:
            raise LsdGpuError("UndistorterPTAM: invalid calibration")
        self.K = K.reshape(3, 3)

    def getK(self) -> np.ndarray:
        return self.K

    def install(self, ctx: "Context"):
        assert (ctx.w, ctx.h) == (self.out_w, self.out_h)
        if self.status == 1:
            ctx._ck(ctx.L.lsdgpu_set_undistorter(ctx.ptr, self.in_w, self.in_h, None, None))
        else:
            ctx._ck(ctx.L.lsdgpu_set_undistorter(ctx.ptr, self.in_w, self.in_h, self.remapX.ctypes.data_as(_fp), self.remapY.ctypes.data_as(_fp)))


def default_track_settings(main_tracker: bool = True) -> TrackSettings:
    s = TrackSettings()
    load().lsdgpu_default_track_settings(C.byref(s))
    if main_tracker:                      # SlamSystem.cpp:80-81
        for lvl in range(4, LEVELS):
            s.maxItsPerLvl[lvl] = 0
    return s


class Context:
    """One device context = the device state of one SlamSystem (frames + one tracker + one depth map)."""

    def __init__(self, w: int, h: int, K: np.ndarray, device: int = 0, max_frames: int = 8, **globals_kw):
        self.L = load()
        self.w, self.h = w, h
        self.K = np.ascontiguousarray(K, np.float32).reshape(3, 3)
        p = _vp()
        rc = self.L.lsdgpu_create(device, w, h, self.K.ctypes.data_as(_fp), max_frames, C.byref(p))
        self.ptr = p
        if rc != 0:
            msg = self.L.lsdgpu_last_error(p).decode() if p else "lsdgpu_create failed"
            if p:
                self.L.lsdgpu_destroy(p)
            self.ptr = None
            raise LsdGpuError(f"lsdgpu_create({w}x{h}) -> {rc}: {msg}")
        if globals_kw:
            self.set_globals(**globals_kw)

    def close(self):
        if getattr(self, "ptr", None):
            self.L.lsdgpu_destroy(self.ptr)
            self.ptr = None

    def __del__(self):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise LsdGpuError(f"rc={rc}: {self.L.lsdgpu_last_error(self.ptr).decode()}")

    def set_globals(self, **kw):
        g = Globals()
        self.L.lsdgpu_default_globals(C.byref(g))
        for k, v in kw.items():
            setattr(g, k, v)
        self._ck(self.L.lsdgpu_set_globals(self.ptr, C.byref(g)))

    def synchronize(self):
        self._ck(self.L.lsdgpu_synchronize(self.ptr))

    def launch_count(self) -> int:
        return int(self.L.lsdgpu_launch_count(self.ptr))

    def timer_begin(self, slot=0):
        self._ck(self.L.lsdgpu_timer_begin(self.ptr, slot))

    def timer_end(self, slot=0) -> None:
        self._ck(self.L.lsdgpu_timer_end(self.ptr, slot))

    def timer_ms(self, slot=0) -> float:
        ms = C.c_float()
        self._ck(self.L.lsdgpu_timer_elapsed_ms(self.ptr, slot, C.byref(ms)))
        return ms.value

    def track_kernel_stats(self, reset=0):
        ms, n, b = C.c_double(), C.c_longlong(), C.c_double()
        self._ck(self.L.lsdgpu_track_kernel_stats(self.ptr, reset, C.byref(ms), C.byref(n), C.byref(b)))
        return ms.value, n.value, b.value

    # ---- Frame ----
    def upload(self, fid: int, image_u8: np.ndarray):
        img = np.ascontiguousarray(image_u8, np.uint8)
        assert img.shape == (self.h, self.w)
        self._ck(self.L.lsdgpu_frame_upload_u8(self.ptr, fid, img.ctypes.data_as(_u8p)))

    def stage_reserve(self, n: int):
        self._ck(self.L.lsdgpu_stage_reserve(self.ptr, n))

    def stage_put(self, index: int, image_u8: np.ndarray):
        img = np.ascontiguousarray(image_u8, np.uint8)
        self._ck(self.L.lsdgpu_stage_put(self.ptr, index, img.ctypes.data_as(_u8p)))

    def frame_from_stage(self, fid: int, index: int):
        self._ck(self.L.lsdgpu_frame_from_stage(self.ptr, fid, index))

    def release(self, fid: int):
        self._ck(self.L.lsdgpu_frame_release(self.ptr, fid))

    def download(self, fid: int, what: int, level: int = 0) -> np.ndarray:
        w, h = self.w >> level, self.h >> level
        if what == BUF_GRADIENTS:
            out = np.empty((h, w, 4), np.float32)
        elif what == BUF_GOODMASK:
            out = np.empty((self.h >> 1, self.w >> 1), np.uint8)
        else:
            out = np.empty((h, w), np.float32)
        self._ck(self.L.lsdgpu_frame_download(self.ptr, fid, what, level, out.ctypes.data_as(_vp)))
        return out

    def set_depth_gt(self, fid: int, depth: np.ndarray, cov_scale: float = 1.0):
        d = np.ascontiguousarray(depth, np.float32)
        self._ck(self.L.lsdgpu_frame_set_depth_gt(self.ptr, fid, d.ctypes.data_as(_fp), cov_scale))

    def set_idepth(self, fid: int, idepth: np.ndarray, var: np.ndarray):
        a = np.ascontiguousarray(idepth, np.float32)
        b = np.ascontiguousarray(var, np.float32)
        self._ck(self.L.lsdgpu_frame_set_idepth(self.ptr, fid, a.ctypes.data_as(_fp), b.ctypes.data_as(_fp)))

    def set_pose(self, fid: int, qts, parent_id: int, initialTrackedResidual: float = 0.0):
        q = np.ascontiguousarray(qts, np.float64)
        self._ck(self.L.lsdgpu_frame_set_pose(self.ptr, fid, q.ctypes.data_as(_dp), parent_id, initialTrackedResidual))

    def get_pose(self, fid: int):
        q = np.zeros(8, np.float64)
        pid, itr = C.c_int(), C.c_float()
        self._ck(self.L.lsdgpu_frame_get_pose(self.ptr, fid, q.ctypes.data_as(_dp), C.byref(pid), C.byref(itr)))
        return q, pid.value, itr.value

    PEER_HANDLE_BYTES = 64

    def peer_export(self) -> bytes:
        """CUDA IPC handle of this context's arena (lsdgpu_peer_export)"""
        buf = C.create_string_buffer(self.PEER_HANDLE_BYTES)
        self._ck(self.L.lsdgpu_peer_export(self.ptr, buf))
        return buf.raw

    def peer_attach(self, rank: int, handles: list):
        """map the arenas of all ranks (handles in rank order) and shard the device-resident tracker over them"""
        blob = b"".join(handles)
        assert len(blob) == self.PEER_HANDLE_BYTES * len(handles)
        self._ck(self.L.lsdgpu_peer_attach(self.ptr, rank, len(handles), C.c_char_p(blob) if len(handles) > 1 else None))

    def peer_detach(self):
        self._ck(self.L.lsdgpu_peer_detach(self.ptr))

    def seq_sum_f32(self, x, valid=None):
        """the sequential fp32 `sum += x[i]` of DepthMap.cpp:1286-1293 through the kernels createKeyFrame uses"""
        x = np.ascontiguousarray(x, np.float32).ravel()
        v = None if valid is None else np.ascontiguousarray(valid, np.uint8).ravel()
        s, c = C.c_float(), C.c_int()
        self._ck(self.L.lsdgpu_seq_sum_f32(self.ptr, x.ctypes.data, None if v is None else v.ctypes.data, x.size, C.byref(s), C.byref(c)))
        return np.float32(s.value), c.value

    def get_counters(self, fid: int):
        a, b = C.c_int(), C.c_int()
        self._ck(self.L.lsdgpu_frame_get_counters(self.ptr, fid, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_counters(self, fid: int, tracked: int, mapped: int):
        self._ck(self.L.lsdgpu_frame_set_counters(self.ptr, fid, tracked, mapped))

    def depth_stats(self, fid: int):
        m, n, f = C.c_float(), C.c_int(), C.c_int()
        self._ck(self.L.lsdgpu_frame_get_depth_stats(self.ptr, fid, C.byref(m), C.byref(n), C.byref(f)))
        return m.value, n.value, bool(f.value)

    def depth_updated_flag(self, fid: int) -> bool:
        """Frame::depthHasBeenUpdatedFlag only (no device sync, unlike depth_stats)."""
        f = C.c_int()
        self._ck(self.L.lsdgpu_frame_get_depth_stats(self.ptr, fid, None, None, C.byref(f)))
        return bool(f.value)

    def undistort(self, raw_u8: np.ndarray) -> np.ndarray:
        """UndistorterPTAM::undistort (Undistorter.cpp:355-411) through the installed tables"""
        raw = np.ascontiguousarray(raw_u8, np.uint8)
        out = np.zeros((self.h, self.w), np.uint8)
        self._ck(self.L.lsdgpu_undistort_u8(self.ptr, raw.ctypes.data_as(C.POINTER(C.c_uint8)), out.ctypes.data_as(C.POINTER(C.c_uint8))))
        return out

    def upload_distorted(self, fid: int, raw_u8: np.ndarray):
        """undistort + Frame construction fused (one H2D copy of the raw image, remap feeds the pyramid kernel)"""
        raw = np.ascontiguousarray(raw_u8, np.uint8)
        self._ck(self.L.lsdgpu_frame_upload_distorted_u8(self.ptr, fid, raw.ctypes.data_as(C.POINTER(C.c_uint8))))

    def pack_pointcloud(self, kf_id: int, level: int = 0) -> np.ndarray:
        """keyframeMsg.pointcloud of ROSOutput3DWrapper::publishKeyframe (ROSOutput3DWrapper.cpp:91-110), packed on the device"""
        n = (self.w >> level) * (self.h >> level)
        out = np.zeros(n, POINT_DENSE)
        self._ck(self.L.lsdgpu_keyframe_pack_pointcloud(self.ptr, kf_id, level, out.ctypes.data_as(_vp)))
        return out

    def export_map(self, kf_ids, cam_to_world_qts, level: int = 0, scaled_th: float = 1e-3, abs_th: float = 1e-1,
                   min_near_support: int = 7):
        """The map as lsd_slam_viewer saves it (KeyFrameDisplay::flushPC over the listed keyframes, lsdgpu_map_export_points):
        returns (points (N, 4) float32 = x, y, z, intensity in world frame, counts per keyframe).  cam_to_world_qts: one
        getScaledCamToWorld() per keyframe as (qx, qy, qz, qw, tx, ty, tz, scale).  Defaults: the ROS viewer parameters
        (cfg/LSDSLAMViewerParams.cfg:20-22); the viewer's built-in defaults are (1, 1, 5) (settings.cpp:36-38)."""
        ids = np.ascontiguousarray(kf_ids, np.int32).reshape(-1)
        qts = np.ascontiguousarray(cam_to_world_qts, np.float64).reshape(-1, 8)
        if qts.shape[0] != ids.size:
            raise ValueError("one camToWorld per keyframe")
        f = MapFilter(scaled_th, abs_th, min_near_support)
        counts = np.zeros(ids.size, np.int32)
        total = C.c_longlong(0)
        args = (self.ptr, ids.size, ids.ctypes.data_as(_ip), qts.ctypes.data_as(_dp), level, C.byref(f))
        self._ck(self.L.lsdgpu_map_export_points(*args, None, 0, counts.ctypes.data_as(_ip), C.byref(total)))
        points = np.empty((total.value, 4), np.float32)
        self._ck(self.L.lsdgpu_map_export_points(*args, points.ctypes.data_as(_vp), total.value, counts.ctypes.data_as(_ip),
                                                 C.byref(total)))
        return points, counts

    def take_reactivation_data(self, kf_id: int):
        self._ck(self.L.lsdgpu_frame_take_reactivation_data(self.ptr, kf_id))

    def reactivation_data(self, kf_id: int):
        """(idepth_reAct, idepthVar_reAct, validity_reAct) of Frame::takeReActivationData (Frame.cpp:107-145)"""
        a, b = np.zeros((self.h, self.w), np.float32), np.zeros((self.h, self.w), np.float32)
        c = np.zeros((self.h, self.w), np.uint8)
        self._ck(self.L.lsdgpu_frame_download_reactivation_data(self.ptr, kf_id, a.ctypes.data_as(_fp), b.ctypes.data_as(_fp),
                                                                c.ctypes.data_as(C.POINTER(C.c_uint8))))
        return a, b, c

    def clear_good_mask(self, fid: int):
        self._ck(self.L.lsdgpu_frame_clear_good_mask(self.ptr, fid))


class SE3Tracker:
    """Mirror of lsd_slam::SE3Tracker (Tracking/SE3Tracker.h): ``trackFrame`` + the public result fields."""

    def __init__(self, ctx: Context, mode: int = 1):
        self.ctx = ctx
        self.mode = mode
        self.settings = default_track_settings()
        self.pointUsage = 0.0
        self.lastGoodCount = self.lastBadCount = 0.0
        self.lastMeanRes = self.lastResidual = 0.0
        self.affineEstimation_a, self.affineEstimation_b = 1.0, 0.0
        self.diverged = False
        self.trackingWasGood = False
        self.last = None

    def importFrame(self, kf_id: int):
        """TrackingReference::importFrame + depthHasBeenUpdatedFlag=false (SlamSystem.cpp:907-912)."""
        self.ctx._ck(self.ctx.L.lsdgpu_ref_import(self.ctx.ptr, kf_id))

    def trackFrame(self, kf_id: int, frame_id: int, frameToReference_initialEstimate) -> np.ndarray:
        q = np.ascontiguousarray(frameToReference_initialEstimate, np.float64)
        r = TrackResult()
        self.ctx._ck(self.ctx.L.lsdgpu_se3_track(self.ctx.ptr, kf_id, frame_id, q.ctypes.data_as(_dp),
                                                 C.byref(self.settings), self.mode, C.byref(r)))
        self.last = r
        self.pointUsage, self.lastGoodCount, self.lastBadCount = r.pointUsage, r.lastGoodCount, r.lastBadCount
        self.lastMeanRes, self.lastResidual = r.lastMeanRes, r.lastResidual
        self.affineEstimation_a, self.affineEstimation_b = r.affineEstimation_a, r.affineEstimation_b
        self.diverged, self.trackingWasGood = bool(r.diverged), bool(r.trackingWasGood)
        return np.array(r.frameToRef_qt, np.float64)

    # ---- permaRef tracking (SURVEY 8f row 2), batched over candidate keyframes ----
    def setPermaRef(self, kf_id: int) -> int:
        n = C.c_int()
        self.ctx._ck(self.ctx.L.lsdgpu_frame_set_perma_ref(self.ctx.ptr, kf_id, C.byref(n)))
        return n.value

    def checkPermaRefOverlap(self, kf_ids, refToFrame_qts) -> np.ndarray:
        ids = np.ascontiguousarray(kf_ids, np.int32)
        q = np.ascontiguousarray(refToFrame_qts, np.float64).reshape(len(ids), 7)
        out = np.zeros(len(ids), np.float32)
        self.ctx._ck(self.ctx.L.lsdgpu_perma_overlap_batch(self.ctx.ptr, len(ids), ids.ctypes.data_as(_ip), q.ctypes.data_as(_dp), out.ctypes.data_as(_fp)))
        return out

    def trackFrameOnPermaref(self, kf_ids, frame_id: int, refToFrame_qts):
        ids = np.ascontiguousarray(kf_ids, np.int32)
        q = np.ascontiguousarray(refToFrame_qts, np.float64).reshape(len(ids), 7)
        res = (TrackResult * len(ids))()
        self.ctx._ck(self.ctx.L.lsdgpu_perma_track_batch(self.ctx.ptr, len(ids), ids.ctypes.data_as(_ip), frame_id, q.ctypes.data_as(_dp), res))
        return list(res)

    def eval(self, kf_id: int, frame_id: int, level: int, refToFrame_qt, a=1.0, b=0.0, write_mask=False) -> EvalResult:
        q = np.ascontiguousarray(refToFrame_qt, np.float32)
        r = EvalResult()
        self.ctx._ck(self.ctx.L.lsdgpu_se3_eval(self.ctx.ptr, kf_id, frame_id, level, q.ctypes.data_as(_fp), a, b,
                                                C.byref(self.settings), int(write_mask), C.byref(r)))
        return r


class Sim3Tracker:
    """Mirror of lsd_slam::Sim3Tracker (Tracking/Sim3Tracker.h:59-160); members as the reference names them."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.settings = default_track_settings(main_tracker=False)     # DenseDepthTrackerSettings(), Sim3Tracker.cpp:57
        self.diverged = False
        self.pointUsage = 0.0
        self.lastResidual = self.lastDepthResidual = self.lastPhotometricResidual = 0.0
        self.affineEstimation_a, self.affineEstimation_b = 1.0, 0.0
        self.lastSim3Hessian = np.zeros((7, 7), np.float32)
        self.last: Sim3Result | None = None

    def trackFrameSim3(self, reference_kf_id: int, frame_id: int, frameToReference_initialEstimate, startLevel: int, finalLevel: int) -> np.ndarray:
        """-> frameToReference as qts[8] (unit quaternion, translation, scale)"""
        q = np.ascontiguousarray(frameToReference_initialEstimate, np.float64)
        r = Sim3Result()
        self.ctx._ck(self.ctx.L.lsdgpu_sim3_track(self.ctx.ptr, reference_kf_id, frame_id, q.ctypes.data_as(_dp), startLevel, finalLevel,
                                                  C.byref(self.settings), C.byref(r)))
        self._take(r)
        return np.array(r.frameToRef_qts)

    def trackFrameSim3Batch(self, reference_kf_ids, frame_ids, inits, startLevel: int, finalLevel: int):
        """n independent trackings in one launch -> list of Sim3Result"""
        a = np.ascontiguousarray(reference_kf_ids, np.int32)
        b = np.ascontiguousarray(frame_ids, np.int32)
        q = np.ascontiguousarray(inits, np.float64).reshape(len(a), 8)
        res = (Sim3Result * len(a))()
        self.ctx._ck(self.ctx.L.lsdgpu_sim3_track_batch(self.ctx.ptr, len(a), a.ctypes.data_as(_ip), b.ctypes.data_as(_ip), q.ctypes.data_as(_dp),
                                                        startLevel, finalLevel, C.byref(self.settings), res))
        return list(res)

    def eval(self, reference_kf_id: int, frame_id: int, level: int, refToFrame_qts, a=1.0, b=0.0) -> Sim3EvalResult:
        q = np.ascontiguousarray(refToFrame_qts, np.float64)
        r = Sim3EvalResult()
        self.ctx._ck(self.ctx.L.lsdgpu_sim3_eval(self.ctx.ptr, reference_kf_id, frame_id, level, q.ctypes.data_as(_dp), a, b,
                                                 C.byref(self.settings), C.byref(r)))
        return r

    def _take(self, r: Sim3Result):
        self.last = r
        self.diverged = bool(r.diverged)
        self.pointUsage = r.pointUsage
        self.lastResidual, self.lastDepthResidual, self.lastPhotometricResidual = r.lastResidual, r.lastDepthResidual, r.lastPhotometricResidual
        self.affineEstimation_a, self.affineEstimation_b = r.affineEstimation_a, r.affineEstimation_b
        self.lastSim3Hessian = np.array(r.lastSim3Hessian, np.float32).reshape(7, 7)


class DepthMap:
    """Mirror of lsd_slam::DepthMap (DepthEstimation/DepthMap.h)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx

    def _ids(self, ids):
        a = np.ascontiguousarray(ids, np.int32)
        return a, a.ctypes.data_as(_ip), len(a)

    def reset(self):
        self.ctx._ck(self.ctx.L.lsdgpu_depth_reset(self.ctx.ptr))

    def isValid(self) -> bool:
        return bool(self.ctx.L.lsdgpu_depth_is_valid(self.ctx.ptr))

    def invalidate(self):
        self.ctx._ck(self.ctx.L.lsdgpu_depth_invalidate(self.ctx.ptr))

    def activeKeyFrame(self) -> int:
        return self.ctx.L.lsdgpu_depth_active_keyframe(self.ctx.ptr)

    def initializeFromGTDepth(self, kf_id: int):
        self.ctx._ck(self.ctx.L.lsdgpu_depth_init_from_gt(self.ctx.ptr, kf_id))

    def setHypotheses(self, kf_id: int, hyp: np.ndarray, reactivated=False, do_set_depth=True):
        a = np.ascontiguousarray(hyp)
        assert a.dtype == HYP_DTYPE
        self.ctx._ck(self.ctx.L.lsdgpu_depth_set_hypotheses(self.ctx.ptr, kf_id, a.ctypes.data_as(C.POINTER(Hyp)),
                                                            int(reactivated), int(do_set_depth)))

    def setFromExistingKF(self, kf_id: int):
        """DepthMap::setFromExistingKF (DepthMap.cpp:920-962) from the keyframe's device-resident reactivation data"""
        self.ctx._ck(self.ctx.L.lsdgpu_depth_set_from_existing_kf(self.ctx.ptr, kf_id))

    def updateKeyframe(self, referenceFrames):
        """DepthMap::updateKeyframe (DepthMap.cpp:1072-1213).  An item is a frame id (tracked on the active keyframe) or a pair
        (frame id, refToKf_qts) for a frame tracked on another keyframe -- refToKf = activeKeyFrame->getScaledCamToWorld().inverse()
        * frame->getScaledCamToWorld() (:1099), which the owner of the pose graph computes."""
        items = list(referenceFrames)
        if all(isinstance(it, (int, np.integer)) for it in items):
            a, p, n = self._ids(items)
            self.ctx._ck(self.ctx.L.lsdgpu_depth_update_keyframe(self.ctx.ptr, p, n))
            return
        descs = (RefDesc * len(items))()
        for d, it in zip(descs, items):
            if isinstance(it, (int, np.integer)):
                d.frame_id, d.tracked_on_kf = int(it), 1
            else:
                d.frame_id, d.tracked_on_kf = int(it[0]), 0
                d.refToKf_qts[:] = [float(v) for v in it[1]]
        self.ctx._ck(self.ctx.L.lsdgpu_depth_update_keyframe_refs(self.ctx.ptr, descs, len(items)))

    def createKeyFrame(self, new_kf_id: int) -> np.ndarray:
        q = np.zeros(8, np.float64)
        self.ctx._ck(self.ctx.L.lsdgpu_depth_create_keyframe(self.ctx.ptr, new_kf_id, q.ctypes.data_as(_dp)))
        return q

    def finalizeKeyFrame(self):
        self.ctx._ck(self.ctx.L.lsdgpu_depth_finalize_keyframe(self.ctx.ptr))

    def observeDepth(self, referenceFrames):
        a, p, n = self._ids(referenceFrames)
        self.ctx._ck(self.ctx.L.lsdgpu_depth_observe(self.ctx.ptr, p, n))

    def regularizeFillHoles(self):
        self.ctx._ck(self.ctx.L.lsdgpu_depth_regularize_fill_holes(self.ctx.ptr))

    def regularize(self, removeOcclusions: bool, validityTH: int = 24):
        self.ctx._ck(self.ctx.L.lsdgpu_depth_regularize(self.ctx.ptr, int(removeOcclusions), validityTH))

    def propagateDepth(self, new_kf_id: int):
        self.ctx._ck(self.ctx.L.lsdgpu_depth_propagate(self.ctx.ptr, new_kf_id))

    def current(self) -> np.ndarray:
        out = np.zeros((self.ctx.h, self.ctx.w), HYP_DTYPE)
        self.ctx._ck(self.ctx.L.lsdgpu_depth_download(self.ctx.ptr, out.ctypes.data_as(C.POINTER(Hyp))))
        return out

    def integral(self) -> np.ndarray:
        out = np.zeros((self.ctx.h, self.ctx.w), np.int32)
        self.ctx._ck(self.ctx.L.lsdgpu_depth_download_integral(self.ctx.ptr, out.ctypes.data_as(C.POINTER(C.c_int32))))
        return out
