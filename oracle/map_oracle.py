"""oracle/map_oracle.py -- the map-export checker (TEST INFRASTRUCTURE; the product never imports it).

Two libraries behind one C name, lsdo_map_export (lsd_slam_viewer's KeyFrameDisplay::flushPC on one keyframeMsg):
    oracle/liblsd_oracle_map.so        the plain-C restatement oracle/lsd_oracle_map.c (gcc, strict IEEE fp32, no FMA
                                       contraction -- the flags of liblsd_oracle.so)
    oracle/_ref/liblsd_ref_viewer.so   lsd_slam_viewer/src/KeyFrameDisplay.cpp + settings.cpp compiled UNMODIFIED from the
                                       reference tree against the stand-in headers of oracle/ref_shim/ (GL no-ops, QGLViewer,
                                       ros/package.h, the keyframeMsg class), with the viewer's own Sophus copy and
                                       oracle/ref_viewer_driver.cpp.  Scalar strict-IEEE flags like liblsd_ref.so.  No
                                       sanitizers: flushPC frees its buffer with a mismatched `delete` (KeyFrameDisplay.cpp:336).
                                       Built only where the reference tree exists; elsewhere a prebuilt copy is used if present.
tests/test_map_export_pin.py holds the restatement to the viewer library's records (tests/golden/ref_map_export_320x240.json,
written by tests/golden/make_map_export_golden.py).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SHIM = os.path.join(HERE, "ref_shim")
ORACLE_SRC = os.path.join(HERE, "lsd_oracle_map.c")
ORACLE_LIB = os.path.join(HERE, "liblsd_oracle_map.so")
VIEWER = "/root/reference/lsd_slam_viewer"
VIEWER_SOURCES = ["src/KeyFrameDisplay.cpp", "src/settings.cpp"]
VIEWER_LIB = os.path.join(HERE, "_ref", "liblsd_ref_viewer.so")
VIEWER_FLAGS = ["-std=gnu++17", "-DNDEBUG", "-fPIC", "-w", f"-I{SHIM}", f"-I{VIEWER}/src", f"-I{VIEWER}/thirdparty/Sophus",
                "-O2", "-ffp-contract=off", "-fno-fast-math", "-msse2"]

# InputPointDense (ROSOutput3DWrapper.h:34-39), one record of keyframeMsg.pointcloud
POINT_DENSE = np.dtype([("idepth", np.float32), ("idepth_var", np.float32), ("color", np.uint8, (4,))])


def viewer_available() -> bool:
    return all(os.path.exists(os.path.join(VIEWER, s)) for s in VIEWER_SOURCES)


def _viewer_deps():
    d = [os.path.join(HERE, "ref_viewer_driver.cpp"), os.path.abspath(__file__)]
    for sub in ("GL", "QGLViewer", "ros", "lsd_slam_viewer", "Eigen"):
        for root, _, files in os.walk(os.path.join(SHIM, sub)):
            d += [os.path.join(root, f) for f in files]
    return d


def _stale(out, deps):
    return not os.path.exists(out) or any(os.path.getmtime(p) > os.path.getmtime(out) for p in deps)


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd[:2])} ... failed:\n{r.stdout}{r.stderr}")


def build(force: bool = False) -> None:
    """Compile the C restatement and, where the reference tree exists, the viewer library."""
    if force or _stale(ORACLE_LIB, [ORACLE_SRC]):
        _run(["gcc", "-std=gnu11", "-fPIC", "-shared", "-Wall", "-O2", "-ffp-contract=off", "-fno-fast-math", "-msse2",
              "-o", ORACLE_LIB, ORACLE_SRC, "-lm"])
    if viewer_available() and (force or _stale(VIEWER_LIB, _viewer_deps())):
        os.makedirs(os.path.dirname(VIEWER_LIB), exist_ok=True)
        _run(["g++"] + VIEWER_FLAGS + ["-shared", "-o", VIEWER_LIB] + [os.path.join(VIEWER, s) for s in VIEWER_SOURCES]
             + [os.path.join(HERE, "ref_viewer_driver.cpp")])


_libs: dict = {}


def lib(flavour=False):
    """False: the C restatement; "ref_viewer": the viewer's own code"""
    path = VIEWER_LIB if flavour == "ref_viewer" else ORACLE_LIB
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        build()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is not built and the reference viewer sources are not available to build it")
    L = C.CDLL(path)
    L.lsdo_map_export.restype = C.c_int
    L.lsdo_map_export.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_double), C.c_float,
                                  C.c_float, C.c_int, C.POINTER(C.c_float)]
    _libs[path] = L
    return L


def map_export(records: np.ndarray, w: int, h: int, fxfycxcy, cam_to_world_qts, scaled_th: float, abs_th: float,
               min_near_support: int, flavour=False) -> np.ndarray:
    """KeyFrameDisplay::flushPC on one keyframe's InputPointDense records: the kept points as (N, 4) float32
    (x, y, z, intensity) in world frame."""
    rec = np.ascontiguousarray(records, POINT_DENSE)
    assert rec.size == w * h
    cam = np.ascontiguousarray(fxfycxcy, np.float32)
    qts = np.ascontiguousarray(cam_to_world_qts, np.float64)
    assert cam.size == 4 and qts.size == 8
    out = np.empty((w * h, 4), np.float32)
    n = lib(flavour).lsdo_map_export(rec.ctypes.data_as(C.c_void_p), w, h, cam.ctypes.data_as(C.POINTER(C.c_float)),
                                     qts.ctypes.data_as(C.POINTER(C.c_double)), scaled_th, abs_th, min_near_support,
                                     out.ctypes.data_as(C.POINTER(C.c_float)))
    if n < 0:
        raise RuntimeError("lsdo_map_export failed")
    return out[:n].copy()


if __name__ == "__main__":
    build(force=True)
    print(ORACLE_LIB, os.path.exists(ORACLE_LIB), VIEWER_LIB, os.path.exists(VIEWER_LIB))
