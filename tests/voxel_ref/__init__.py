"""ctypes view of the CPU references of D2PC_FILTER_VOXEL (test infrastructure, not product code).

voxel_grid()      tests/voxel_ref/voxel_grid.c: the recipe of include/d2pc_b200.h, summation in ascending point
                  index -- what the GPU must reproduce bit for bit.
voxel_pcl_order() tests/voxel_ref/pcl_order.cpp: PCL's applyFilter with its own std::sort order (no limit field).

Both are compiled on first use into a per-user temporary directory keyed by the sources' hash, so the repository
tree is never written.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = {"voxel_grid.c": ["gcc", "-std=c11"], "pcl_order.cpp": ["g++", "-std=c++14"]}
_libs: dict[str, C.CDLL] = {}

FIELDS = {None: -1, "x": 0, "y": 1, "z": 2}


def _lib(src: str) -> C.CDLL:
    if src in _libs:
        return _libs[src]
    path = os.path.join(_HERE, src)
    digest = hashlib.sha256(open(path, "rb").read()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"d2pc_voxel_ref_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"{os.path.splitext(src)[0]}_{digest}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        compiler, std = _SOURCES[src]
        subprocess.run([compiler, std, "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Werror", path,
                        "-o", tmp, "-lm"], check=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    fp = C.POINTER(C.c_float)
    if src == "voxel_grid.c":
        lib.d2pc_voxel_ref.argtypes = [fp, C.c_size_t, C.c_float, C.c_float, C.c_float, C.c_uint32, C.c_int,
                                       C.c_double, C.c_double, fp, C.POINTER(C.c_int)]
        lib.d2pc_voxel_ref.restype = C.c_size_t
    else:
        lib.d2pc_voxel_pcl_order.argtypes = [fp, C.c_size_t, C.c_float, C.c_float, C.c_float, C.c_uint32, fp,
                                             C.POINTER(C.c_int)]
        lib.d2pc_voxel_pcl_order.restype = C.c_size_t
    _libs[src] = lib
    return lib


def _leaves(leaf):
    return (leaf, leaf, leaf) if np.isscalar(leaf) else tuple(leaf)


def _cloud(cloud) -> np.ndarray:
    return np.ascontiguousarray(np.frombuffer(np.ascontiguousarray(cloud).tobytes(), np.float32).reshape(-1, 4))


def voxel_grid(cloud, leaf, min_points: int = 0, limit=None) -> tuple[bytes, int]:
    """cloud: CROP cloud bytes (N*16).  limit: None or (field, lo, hi).  -> (PointCloud2.data bytes, is_dense)."""
    pts = _cloud(cloud)
    out = np.empty(max(len(pts), 1) * 4, np.float32)
    dense = C.c_int(0)
    field, lo, hi = (None, 0.0, 0.0) if limit is None else limit
    fp = C.POINTER(C.c_float)
    k = _lib("voxel_grid.c").d2pc_voxel_ref(pts.ctypes.data_as(fp), len(pts), *_leaves(leaf), int(min_points),
                                            FIELDS[field], float(lo), float(hi), out.ctypes.data_as(fp), C.byref(dense))
    return out[: 4 * k].tobytes(), dense.value


def voxel_pcl_order(cloud, leaf, min_points: int = 0) -> tuple[bytes, int]:
    pts = _cloud(cloud)
    out = np.empty(max(len(pts), 1) * 4, np.float32)
    dense = C.c_int(0)
    fp = C.POINTER(C.c_float)
    k = _lib("pcl_order.cpp").d2pc_voxel_pcl_order(pts.ctypes.data_as(fp), len(pts), *_leaves(leaf), int(min_points),
                                                   out.ctypes.data_as(fp), C.byref(dense))
    return out[: 4 * k].tobytes(), dense.value
