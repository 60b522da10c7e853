"""ctypes view of the CPU references of the projected 2-D map (test infrastructure, not product code).

ProjTree            tests/map_ref/projected_map.cpp: octree.PointerTree (the file includes octree_pointer.cpp) plus
                    octomap_server's /projected_map restated literally, and a tree built from (key, log-odds) pairs.
projected_map()     tests/map_ref/projected_map.c: the header's per-voxel recipe from Morton-sorted flat voxels.

Both return (cells (height, width) int8, resolution float, (origin_x, origin_y)), None when octomap_server publishes
nothing (an empty tree), or the string "BAD_DIMS" when a padded corner has no key.  Compiled like octree.py's sources,
into a per-user temporary directory keyed by their hash, so the repository tree is never written.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import sys
import tempfile

import numpy as np

from map_ref import logodds, octree

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "disparity_to_point_cloud_b200", "csrc")
_SOURCES = {"projected_map.cpp": (["g++", "-std=c++14"], ["octree_pointer.cpp", "octomap_literal.cpp"]),
            "projected_map.c": (["gcc", "-std=c11"], [])}
_libs: dict[str, C.CDLL] = {}
_FP, _U64P, _VP, _DP = C.POINTER(C.c_float), C.POINTER(C.c_uint64), C.c_void_p, C.POINTER(C.c_double)
_U32P = C.POINTER(C.c_uint32)
BIG = sys.float_info.max


def _lib(src: str) -> C.CDLL:
    if src in _libs:
        return _libs[src]
    cc, deps = _SOURCES[src]
    path = os.path.join(_HERE, src)
    h = hashlib.sha256(open(path, "rb").read())
    h.update(open(os.path.join(_CSRC, "map_math.h"), "rb").read())
    for dep in deps:
        h.update(open(os.path.join(_HERE, dep), "rb").read())
    out_dir = os.path.join(tempfile.gettempdir(), f"d2pc_map_ref_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"{os.path.splitext(src)[0]}_{os.path.splitext(src)[1][1:]}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(cc + ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Werror", "-I", _CSRC, path,
                             "-o", tmp, "-lm"], check=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    if src == "projected_map.cpp":
        base = octree._lib("octree_pointer.cpp")  # the same ptr_* entries, compiled into this library too
        for name in ("ptr_new", "ptr_free", "ptr_clear", "ptr_set_params", "ptr_insert", "ptr_update", "ptr_write",
                     "ptr_voxels", "ptr_tree_size", "ptr_load_full"):
            f, g = getattr(lib, name), getattr(base, name)
            f.argtypes, f.restype = g.argtypes, g.restype
        lib.ptr_set_values.argtypes, lib.ptr_set_values.restype = [_VP, _U64P, _FP, C.c_size_t], None
        lib.ptr_projected_map.argtypes = [_VP] + [C.c_double] * 4 + [_U32P, _U32P, _FP, _DP]
        lib.ptr_projected_map.restype = C.c_int
        lib.ptr_projected_cells.argtypes, lib.ptr_projected_cells.restype = [C.c_void_p], None
    else:
        lib.d2pc_projected_map_ref.argtypes = [_U64P, _U32P, C.c_size_t, C.c_double, C.c_float] + [C.c_double] * 4 + \
            [C.c_void_p, C.c_uint64, _U32P, _U32P, _DP]
        lib.d2pc_projected_map_ref.restype = C.c_int
    _libs[src] = lib
    return lib


class ProjTree(octree.PointerTree):
    """octree.PointerTree on projected_map.cpp's copy of it, plus projected_map() and set_values()."""

    def __init__(self, **params):
        self._L = _lib("projected_map.cpp")
        p = dict(params)
        self.resolution = p.pop("resolution", 0.05)
        self._h = self._L.ptr_new(self.resolution)
        self.set_params(**p)

    def set_values(self, keys, log_odds):
        """The tree setNodeValue builds from (n, 3) uint16 keys and their float32 log-odds, in that order."""
        k = octree._pack(keys)
        lo = np.ascontiguousarray(log_odds, np.float32)
        self._L.ptr_set_values(self._h, k.ctypes.data_as(_U64P), lo.ctypes.data_as(_FP), len(k))

    def projected_map(self, occupancy_min_z=-BIG, occupancy_max_z=BIG, min_x_size=0.0, min_y_size=0.0):
        w, h, res, origin = C.c_uint32(), C.c_uint32(), C.c_float(), (C.c_double * 2)()
        rc = self._L.ptr_projected_map(self._h, occupancy_min_z, occupancy_max_z, min_x_size, min_y_size, C.byref(w),
                                       C.byref(h), C.byref(res), origin)
        if rc == 1:
            return None
        if rc == -3:
            return "BAD_DIMS"
        cells = np.empty(w.value * h.value, np.int8)
        self._L.ptr_projected_cells(cells.ctypes.data)
        return cells.reshape(h.value, w.value), res.value, (origin[0], origin[1])


def projected_map(keys, log_odds, resolution, occupancy_thres=0.5, occupancy_min_z=-BIG, occupancy_max_z=BIG,
                  min_x_size=0.0, min_y_size=0.0):
    """The per-voxel recipe on the known voxels in Morton order ((n, 3) uint16 keys, float32 log-odds)."""
    k = octree._pack(keys)
    lo = np.ascontiguousarray(log_odds, np.float32).view(np.uint32)
    f = _lib("projected_map.c").d2pc_projected_map_ref
    w, h, origin = C.c_uint32(), C.c_uint32(), (C.c_double * 2)()
    args = (k.ctypes.data_as(_U64P), lo.ctypes.data_as(_U32P), len(k), resolution, logodds(occupancy_thres),
            occupancy_min_z, occupancy_max_z, min_x_size, min_y_size)
    rc = f(*args, None, 0, C.byref(w), C.byref(h), origin)
    if rc == -3:
        return "BAD_DIMS"
    assert rc == 0, rc
    if len(k) == 0:
        return None
    cells = np.empty(max(w.value * h.value, 1), np.int8)
    assert f(*args, cells.ctypes.data, len(cells), C.byref(w), C.byref(h), origin) == 0
    return cells[:w.value * h.value].reshape(h.value, w.value), float(np.float32(resolution)), (origin[0], origin[1])
