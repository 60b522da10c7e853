"""ctypes view of the CPU references of the laser scan output (test infrastructure, not product code).

scan()        tests/scan_ref/scan.c: the recipe of include/d2pc_b200.h, with the library's csrc/scan_math.h.
p2l()         tests/scan_ref/p2l_cloudcb.cpp: PointCloudToLaserScanNodelet::cloudCb restated literally (glibc hypot and
              atan2, float message fields, a sequential min).
angle(), rng  the shared math of csrc/scan_math.h on one input, as the kernel computes it.

scan() and p2l() take a cloud of 16-byte points and the params as keywords (the nodelet's names, the library's
defaults) and return the float32 ranges.  The sources are compiled on first use into a per-user temporary directory
keyed by their hash, so the repository tree is never written.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import math
import os
import subprocess
import sys
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "disparity_to_point_cloud_b200", "csrc")
_SOURCES = {"scan.c": ["gcc", "-std=c11"], "p2l_cloudcb.cpp": ["g++", "-std=c++14"]}
_libs: dict[str, C.CDLL] = {}
_FP, _DP = C.POINTER(C.c_float), C.POINTER(C.c_double)

# the nodelet's defaults as the library states them (include/d2pc_b200.h)
DEFAULTS = dict(min_height=sys.float_info.min, max_height=sys.float_info.max, angle_min=-math.pi, angle_max=math.pi,
                angle_increment=math.pi / 180.0, scan_time=1.0 / 30.0, range_min=0.0, range_max=sys.float_info.max,
                use_inf=1, inf_epsilon=1.0)


def _lib(src: str) -> C.CDLL:
    if src in _libs:
        return _libs[src]
    path = os.path.join(_HERE, src)
    h = hashlib.sha256(open(path, "rb").read())
    h.update(open(os.path.join(_CSRC, "scan_math.h"), "rb").read())
    out_dir = os.path.join(tempfile.gettempdir(), f"d2pc_scan_ref_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"{os.path.splitext(src)[0]}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(_SOURCES[src] + ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Werror", "-I", _CSRC,
                                        path, "-o", tmp, "-lm"], check=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    if src == "scan.c":
        lib.d2pc_scan_angle_ref.argtypes, lib.d2pc_scan_angle_ref.restype = [C.c_double, C.c_double], C.c_double
        lib.d2pc_scan_range_ref.argtypes, lib.d2pc_scan_range_ref.restype = [C.c_float, C.c_float], C.c_double
    _libs[src] = lib
    return lib


def params(**kw) -> dict:
    p = dict(DEFAULTS)
    for k, v in kw.items():
        if k not in p and k != "keep_cloud":
            raise ValueError(f"unknown scan param {k!r}")
        p[k] = v
    return p


def _run(src: str, fn: str, cloud, kw) -> np.ndarray:
    p = params(**kw)
    pts = np.ascontiguousarray(np.frombuffer(np.ascontiguousarray(cloud).tobytes(), np.float32).reshape(-1, 4))
    prm = np.array([p[k] for k in ("min_height", "max_height", "angle_min", "angle_max", "angle_increment",
                                   "range_min", "range_max", "inf_epsilon")], np.float64)
    f = getattr(_lib(src), fn)
    f.argtypes, f.restype = [_FP, C.c_size_t, _DP, C.c_int, _FP, C.c_uint32], C.c_uint32
    n = f(pts.ctypes.data_as(_FP), len(pts), prm.ctypes.data_as(_DP), int(p["use_inf"]), None, 0)
    out = np.empty(n, np.float32)
    f(pts.ctypes.data_as(_FP), len(pts), prm.ctypes.data_as(_DP), int(p["use_inf"]), out.ctypes.data_as(_FP), n)
    return out


def scan(cloud, **kw) -> np.ndarray:
    return _run("scan.c", "d2pc_laser_scan_ref", cloud, kw)


def p2l(cloud, **kw) -> np.ndarray:
    return _run("p2l_cloudcb.cpp", "d2pc_p2l_cloudcb", cloud, kw)


def fields(**kw) -> dict:
    """The message fields the scan carries: the params rounded to float, time_increment 0."""
    p = params(**kw)
    with np.errstate(over="ignore"):  # range_max DBL_MAX is +inf as a float
        f = {k: float(np.float32(p[k])) for k in ("angle_min", "angle_max", "angle_increment", "scan_time", "range_min",
                                                  "range_max")}
    f["time_increment"] = 0.0
    return f


def angle(y: float, x: float) -> float:
    return _lib("scan.c").d2pc_scan_angle_ref(y, x)


def rng(x: float, y: float) -> float:
    return _lib("scan.c").d2pc_scan_range_ref(x, y)


def math_arrays(x, y):
    """(range, angle) of float32 arrays x, y, as the kernel computes them (float64 arrays)."""
    x, y = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(y, np.float32)
    r, a = np.empty(len(x)), np.empty(len(x))
    f = _lib("scan.c").d2pc_scan_math_ref
    f.argtypes, f.restype = [_FP, _FP, C.c_size_t, _DP, _DP], None
    f(x.ctypes.data_as(_FP), y.ctypes.data_as(_FP), len(x), r.ctypes.data_as(_DP), a.ctypes.data_as(_DP))
    return r, a
