"""ctypes view of the CPU references of the radius outlier stage (test infrastructure, not product code).

radius_outlier()  tests/outlier_ref/radius_outlier.c: the recipe of include/d2pc_b200.h, from a uniform grid
                  (method="grid", the default) or literally over every pair (method="brute").
pcl_knn()         tests/outlier_ref/pcl_branches.cpp: PCL's is_dense branch (k-NN, partial sort).
pcl_radius()      the same file: PCL's radiusSearch branch (strict < against the float radius squared).

Every function takes a cloud of 16-byte points and returns the PointCloud2.data bytes of the kept points (is_dense
is always 1).  The sources are compiled on first use into a per-user temporary directory keyed by their hash, so
the repository tree is never written.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = {"radius_outlier.c": ["gcc", "-std=c11"], "pcl_branches.cpp": ["g++", "-std=c++14"]}
_libs: dict[str, C.CDLL] = {}
_FP = C.POINTER(C.c_float)
_ARGS = [_FP, C.c_size_t, C.c_double, C.c_uint32, _FP]


def _lib(src: str) -> C.CDLL:
    if src in _libs:
        return _libs[src]
    path = os.path.join(_HERE, src)
    digest = hashlib.sha256(open(path, "rb").read()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"d2pc_outlier_ref_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"{os.path.splitext(src)[0]}_{digest}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        compiler, std = _SOURCES[src]
        subprocess.run([compiler, std, "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Werror", path,
                        "-o", tmp, "-lm"], check=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    names = ["d2pc_ror_grid", "d2pc_ror_brute"] if src == "radius_outlier.c" else ["d2pc_ror_pcl_knn",
                                                                                    "d2pc_ror_pcl_radius"]
    for name in names:
        fn = getattr(lib, name)
        fn.argtypes = _ARGS
        fn.restype = C.c_size_t
    _libs[src] = lib
    return lib


def _cloud(cloud) -> np.ndarray:
    return np.ascontiguousarray(np.frombuffer(np.ascontiguousarray(cloud).tobytes(), np.float32).reshape(-1, 4))


def _run(src: str, name: str, cloud, radius: float, min_neighbors: int) -> bytes:
    pts = _cloud(cloud)
    out = np.empty(max(len(pts), 1) * 4, np.float32)
    k = getattr(_lib(src), name)(pts.ctypes.data_as(_FP), len(pts), float(radius), int(min_neighbors),
                                 out.ctypes.data_as(_FP))
    return out[: 4 * k].tobytes()


def radius_outlier(cloud, radius: float, min_neighbors: int = 1, method: str = "grid") -> bytes:
    return _run("radius_outlier.c", {"grid": "d2pc_ror_grid", "brute": "d2pc_ror_brute"}[method], cloud, radius,
                min_neighbors)


def pcl_knn(cloud, radius: float, min_neighbors: int = 1) -> bytes:
    return _run("pcl_branches.cpp", "d2pc_ror_pcl_knn", cloud, radius, min_neighbors)


def pcl_radius(cloud, radius: float, min_neighbors: int = 1) -> bytes:
    return _run("pcl_branches.cpp", "d2pc_ror_pcl_radius", cloud, radius, min_neighbors)
