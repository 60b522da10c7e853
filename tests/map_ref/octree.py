"""ctypes view of the CPU references of the octomap_msgs/Octomap export (test infrastructure, not product code).

PointerTree     tests/map_ref/octree_pointer.cpp: octomap's pointer OcTree (updateNode with pruning) restated
                literally, driven by octomap_literal.cpp's insertScan, and its writeData / writeBinaryData / readData.
read_full()     readData of a full stream into a fresh pointer tree, expanded to full-depth voxels.
octomap_data()  tests/map_ref/octomap_msg.c: the header's octomap_msgs/Octomap recipe from sorted flat voxels.

The sources are compiled on first use into a per-user temporary directory keyed by their hash (and that of the files
they include), so the repository tree is never written.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from map_ref import DEFAULTS, logodds

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "disparity_to_point_cloud_b200", "csrc")
# source -> (compiler, the sources it #includes)
_SOURCES = {"octree_pointer.cpp": (["g++", "-std=c++14"], ["octomap_literal.cpp"]),
            "octomap_msg.c": (["gcc", "-std=c11"], [])}
_libs: dict[str, C.CDLL] = {}
_FP, _U64P, _VP = C.POINTER(C.c_float), C.POINTER(C.c_uint64), C.c_void_p


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
    so = os.path.join(out_dir, f"{os.path.splitext(src)[0]}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(cc + ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Werror", "-I", _CSRC, path,
                             "-o", tmp, "-lm"], check=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    if src == "octree_pointer.cpp":
        lib.ptr_new.argtypes, lib.ptr_new.restype = [C.c_double], _VP
        lib.ptr_free.argtypes, lib.ptr_free.restype = [_VP], None
        lib.ptr_clear.argtypes, lib.ptr_clear.restype = [_VP], None
        lib.ptr_set_params.argtypes = [_VP] + [C.c_double] * 6
        lib.ptr_set_params.restype = None
        lib.ptr_insert.argtypes = [_VP, _FP, C.c_size_t, C.c_float, C.c_float, C.c_float]
        lib.ptr_insert.restype = None
        lib.ptr_update.argtypes = [_VP, C.c_uint16, C.c_uint16, C.c_uint16, C.c_int]
        lib.ptr_update.restype = None
        lib.ptr_write.argtypes, lib.ptr_write.restype = [_VP, C.c_int, C.POINTER(C.c_void_p)], C.c_size_t
        lib.ptr_voxels.argtypes = [_VP, _U64P, _FP, C.c_size_t, C.POINTER(C.c_uint)]
        lib.ptr_voxels.restype = C.c_size_t
        lib.ptr_tree_size.argtypes, lib.ptr_tree_size.restype = [_VP], C.c_size_t
        lib.ptr_load_full.argtypes, lib.ptr_load_full.restype = [_VP, C.c_char_p, C.c_size_t], None
        lib.ptr_read_full.argtypes = [C.c_char_p, C.c_size_t, _U64P, _FP, C.c_size_t, C.POINTER(C.c_size_t)]
        lib.ptr_read_full.restype = C.c_size_t
    else:
        lib.d2pc_octomap_ref.argtypes = [_U64P, C.POINTER(C.c_uint32), C.c_size_t, C.c_int, C.c_float, C.c_void_p,
                                         C.c_size_t]
        lib.d2pc_octomap_ref.restype = C.c_size_t
    _libs[src] = lib
    return lib


def _unpack(keys):
    return np.stack([(keys >> np.uint64(16 * a)) & np.uint64(0xFFFF) for a in range(3)], 1).astype(np.uint16)


def _pack(keys):
    k = np.asarray(keys, np.uint64).reshape(-1, 3)
    return np.ascontiguousarray(k[:, 0] | (k[:, 1] << np.uint64(16)) | (k[:, 2] << np.uint64(32)))


class PointerTree:
    """octomap's pointer OcTree with pruning (octree_pointer.cpp), the same interface as Octree for inserts, plus
    update() for single updateNode calls, the serializers and the tree's shape."""

    def __init__(self, **params):
        p = dict(DEFAULTS)
        p.update(params)
        self._L = _lib("octree_pointer.cpp")
        self.resolution = p["resolution"]
        self._h = self._L.ptr_new(self.resolution)
        self.set_params(**{k: v for k, v in p.items() if k != "resolution"})

    def set_params(self, **params):
        p = dict(DEFAULTS)
        p.update(getattr(self, "_params", {}))
        p.update(params)
        self._params = {k: v for k, v in p.items() if k != "resolution"}
        self._L.ptr_set_params(self._h, p["prob_hit"], p["prob_miss"], p["clamp_min"], p["clamp_max"],
                               p["occupancy_thres"], p["max_range"])

    def clear(self):
        self._L.ptr_clear(self._h)

    def insert(self, cloud, origin=(0.0, 0.0, 0.0)):
        pts = np.ascontiguousarray(np.frombuffer(np.ascontiguousarray(cloud).tobytes(), np.float32).reshape(-1, 4))
        o = np.asarray(origin, np.float32)
        self._L.ptr_insert(self._h, pts.ctypes.data_as(_FP), len(pts), float(o[0]), float(o[1]), float(o[2]))

    def update(self, key, occupied: bool):
        """One OccupancyOcTreeBase::updateNode(key, occupied)."""
        self._L.ptr_update(self._h, int(key[0]), int(key[1]), int(key[2]), 1 if occupied else 0)

    def data(self, binary: bool = False) -> bytes:
        """writeData (the full format) or writeBinaryData."""
        p = C.c_void_p()
        n = self._L.ptr_write(self._h, 1 if binary else 0, C.byref(p))
        return C.string_at(p, n) if n else b""

    def voxels(self, leaf_depths=None):
        """The tree expanded to full-depth voxels in pre-order: (keys (n, 3) uint16, log-odds float32).  leaf_depths:
        a list that receives the number of leaves at each depth 0..16."""
        depths = (C.c_uint * 17)()
        n = self._L.ptr_voxels(self._h, None, None, 0, None)
        keys, lo = np.empty(max(n, 1), np.uint64), np.empty(max(n, 1), np.float32)
        self._L.ptr_voxels(self._h, keys.ctypes.data_as(_U64P), lo.ctypes.data_as(_FP), n, depths)
        if leaf_depths is not None:
            leaf_depths[:] = list(depths)
        return _unpack(keys[:n]), lo[:n]

    def load(self, full: bytes):
        """readData of a full stream: the tree becomes the one it describes."""
        self._L.ptr_load_full(self._h, full, len(full))

    def tree_size(self) -> int:
        return int(self._L.ptr_tree_size(self._h))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._L.ptr_free(h)
            self._h = None


def read_full(data: bytes):
    """readData of a full stream into a fresh pointer tree, expanded to (keys (n, 3) uint16, log-odds float32); the
    stream must be read exactly."""
    L = _lib("octree_pointer.cpp")
    used = C.c_size_t()
    n = L.ptr_read_full(data, len(data), None, None, 0, C.byref(used))
    keys, lo = np.empty(max(n, 1), np.uint64), np.empty(max(n, 1), np.float32)
    L.ptr_read_full(data, len(data), keys.ctypes.data_as(_U64P), lo.ctypes.data_as(_FP), n, C.byref(used))
    assert used.value == len(data), (used.value, len(data))
    return _unpack(keys[:n]), lo[:n]


def octomap_data(keys, log_odds, binary: bool = False, occupancy_thres: float = 0.5) -> bytes:
    """The recipe's data of the known voxels in Morton order ((n, 3) uint16 keys, float32 log-odds)."""
    k = _pack(keys)
    lo = np.ascontiguousarray(log_odds, np.float32).view(np.uint32)
    f = _lib("octomap_msg.c").d2pc_octomap_ref
    thres = logodds(occupancy_thres)
    n = f(k.ctypes.data_as(_U64P), lo.ctypes.data_as(C.POINTER(C.c_uint32)), len(k), int(binary), thres, None, 0)
    out = np.zeros(max(n, 1), np.uint8)
    got = f(k.ctypes.data_as(_U64P), lo.ctypes.data_as(C.POINTER(C.c_uint32)), len(k), int(binary), thres,
            out.ctypes.data, n)
    assert got == n
    return out[:n].tobytes()
