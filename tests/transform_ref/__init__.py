"""ctypes view of the CPU references of the cloud transform stage (test infrastructure, not product code).

transform()  tests/transform_ref/transform.c: the recipe of include/d2pc_b200.h.
pcl()        tests/transform_ref/pcl_transform.cpp: transformPointCloud's dense and non-dense loops restated literally
             with the scalar Transformer's row order.
pcl_sse()    the same loops with the SSE2 Transformer's row order, x*c0 + (y*c1 + (z*c2 + c3)).

Each takes a cloud of 16-byte points and a 3x4 matrix and returns the PointCloud2.data bytes of the transformed cloud
(same point count).  The sources are compiled on first use into a per-user temporary directory keyed by their hash,
so the repository tree is never written.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = {"transform.c": ["gcc", "-std=c11"], "pcl_transform.cpp": ["g++", "-std=c++14"]}
_libs: dict[str, C.CDLL] = {}
_FP = C.POINTER(C.c_float)
IDENTITY = np.eye(3, 4, dtype=np.float32)


def _lib(src: str) -> C.CDLL:
    if src in _libs:
        return _libs[src]
    path = os.path.join(_HERE, src)
    digest = hashlib.sha256(open(path, "rb").read()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"d2pc_transform_ref_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"{os.path.splitext(src)[0]}_{digest}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(_SOURCES[src] + ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Werror", path,
                                        "-o", tmp, "-lm"], check=True)
        os.replace(tmp, so)
    _libs[src] = C.CDLL(so)
    return _libs[src]


def _points(cloud) -> np.ndarray:
    return np.ascontiguousarray(np.frombuffer(np.ascontiguousarray(cloud).tobytes(), np.float32).reshape(-1, 4))


def _matrix(m) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(m, np.float32).reshape(12))


def transform(cloud, matrix) -> bytes:
    pts, m = _points(cloud), _matrix(matrix)
    out = np.empty_like(pts)
    fn = _lib("transform.c").d2pc_transform_ref
    fn.argtypes, fn.restype = [_FP, C.c_size_t, _FP, _FP], None
    fn(pts.ctypes.data_as(_FP), len(pts), m.ctypes.data_as(_FP), out.ctypes.data_as(_FP))
    return out.tobytes()


def _pcl(name: str, cloud, matrix, is_dense: bool) -> bytes:
    pts, m = _points(cloud), _matrix(matrix)
    out = np.empty_like(pts)
    fn = getattr(_lib("pcl_transform.cpp"), name)
    fn.argtypes, fn.restype = [_FP, C.c_size_t, C.c_int, _FP, _FP], None
    fn(pts.ctypes.data_as(_FP), len(pts), 1 if is_dense else 0, m.ctypes.data_as(_FP), out.ctypes.data_as(_FP))
    return out.tobytes()


def pcl(cloud, matrix, is_dense: bool = False) -> bytes:
    return _pcl("d2pc_transform_pcl", cloud, matrix, is_dense)


def pcl_sse(cloud, matrix, is_dense: bool = False) -> bytes:
    return _pcl("d2pc_transform_pcl_sse", cloud, matrix, is_dense)
