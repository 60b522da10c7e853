"""ctypes view of the CPU references of the occupancy map (test infrastructure, not product code).

ray() / rays_digest()   tests/map_ref/occupancy.c: the header's recipe per ray, on the library's csrc/map_math.h.
Octree                  tests/map_ref/octomap_literal.cpp: OctomapServer::insertScan, computeRayKeys and
                        OcTree::updateNode restated literally (unordered_set key sets, a map of full-depth leaves).
literal_rays_digest()   the same per-ray digest from the literal restatement.

The sources are compiled on first use into a per-user temporary directory keyed by their hash, so the repository tree
is never written.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "disparity_to_point_cloud_b200", "csrc")
_SOURCES = {"occupancy.c": ["gcc", "-std=c11"], "octomap_literal.cpp": ["g++", "-std=c++14"]}
_libs: dict[str, C.CDLL] = {}
_FP, _U16P, _U64P, _VP = C.POINTER(C.c_float), C.POINTER(C.c_uint16), C.POINTER(C.c_uint64), C.c_void_p

# octomap_server's defaults as the library states them (include/d2pc_b200.h)
DEFAULTS = dict(resolution=0.05, prob_hit=0.7, prob_miss=0.4, clamp_min=0.12, clamp_max=0.97, occupancy_thres=0.5,
                max_range=-1.0)


def _lib(src: str) -> C.CDLL:
    if src in _libs:
        return _libs[src]
    path = os.path.join(_HERE, src)
    h = hashlib.sha256(open(path, "rb").read())
    h.update(open(os.path.join(_CSRC, "map_math.h"), "rb").read())
    out_dir = os.path.join(tempfile.gettempdir(), f"d2pc_map_ref_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"{os.path.splitext(src)[0]}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(_SOURCES[src] + ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Werror", "-I", _CSRC,
                                        path, "-o", tmp, "-lm"], check=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    if src == "occupancy.c":
        lib.d2pc_map_ray_ref.argtypes = [_FP, _FP, C.c_double, C.c_double, _U16P, C.c_uint32, _U16P,
                                         C.POINTER(C.c_int)]
        lib.d2pc_map_ray_ref.restype = C.c_uint32
        lib.d2pc_map_rays_digest.argtypes = [_FP, C.c_size_t, C.c_double, C.c_double, _U64P]
        lib.d2pc_map_rays_digest.restype = None
        lib.d2pc_map_morton_ref.argtypes = [C.c_uint16, C.c_uint16, C.c_uint16]
        lib.d2pc_map_morton_ref.restype = C.c_uint64
    else:
        lib.oct_new.argtypes, lib.oct_new.restype = [C.c_double], _VP
        lib.oct_free.argtypes, lib.oct_free.restype = [_VP], None
        lib.oct_clear.argtypes, lib.oct_clear.restype = [_VP], None
        lib.oct_set_params.argtypes = [_VP] + [C.c_double] * 6
        lib.oct_set_params.restype = None
        lib.oct_logodds.argtypes, lib.oct_logodds.restype = [C.c_double], C.c_float
        lib.oct_insert.argtypes = [_VP, _FP, C.c_size_t, C.c_float, C.c_float, C.c_float]
        lib.oct_insert.restype = None
        lib.oct_voxels.argtypes, lib.oct_voxels.restype = [_VP, _U64P, _FP, C.c_size_t], C.c_size_t
        lib.oct_centers.argtypes, lib.oct_centers.restype = [_VP, _FP, C.c_size_t], C.c_size_t
        lib.oct_rays_digest.argtypes = [_FP, C.c_size_t, C.c_double, C.c_double, _U64P]
        lib.oct_rays_digest.restype = None
    _libs[src] = lib
    return lib


def ray(origin, point, resolution=0.05, max_range=-1.0):
    """The recipe's cells of one point: (free keys as an (m, 3) uint16 array in DDA order, occupied key or None)."""
    o, p = np.asarray(origin, np.float32), np.asarray(point, np.float32)
    hit, valid = np.zeros(3, np.uint16), C.c_int()
    f = _lib("occupancy.c").d2pc_map_ray_ref
    n = f(o.ctypes.data_as(_FP), p.ctypes.data_as(_FP), resolution, max_range, None, 0,
          hit.ctypes.data_as(_U16P), C.byref(valid))
    keys = np.zeros((max(n, 1), 3), np.uint16)
    f(o.ctypes.data_as(_FP), p.ctypes.data_as(_FP), resolution, max_range, keys.ctypes.data_as(_U16P), n,
      hit.ctypes.data_as(_U16P), C.byref(valid))
    return keys[:n], (tuple(int(k) for k in hit) if valid.value else None)


def _digest(fn, origins, points, resolution, max_range):
    pairs = np.ascontiguousarray(np.concatenate([np.asarray(origins, np.float32).reshape(-1, 3),
                                                 np.asarray(points, np.float32).reshape(-1, 3)], axis=1))
    out = np.empty((len(pairs), 3), np.uint64)
    fn(pairs.ctypes.data_as(_FP), len(pairs), resolution, max_range, out.ctypes.data_as(_U64P))
    return out


def rays_digest(origins, points, resolution=0.05, max_range=-1.0) -> np.ndarray:
    """(free cell count, FNV-1a of the free keys, packed occupied key or 2^64 - 1) per (origin, point), the recipe."""
    return _digest(_lib("occupancy.c").d2pc_map_rays_digest, origins, points, resolution, max_range)


def literal_rays_digest(origins, points, resolution=0.05, max_range=-1.0) -> np.ndarray:
    """The same digest from the literal restatement of computeRayKeys and insertScan."""
    return _digest(_lib("octomap_literal.cpp").oct_rays_digest, origins, points, resolution, max_range)


def morton(kx: int, ky: int, kz: int) -> int:
    return int(_lib("occupancy.c").d2pc_map_morton_ref(kx, ky, kz))


def logodds(p: float) -> float:
    """octomap's (float)log(p / (1 - p)), as a Python float."""
    return float(_lib("octomap_literal.cpp").oct_logodds(p))


class Octree:
    """The literal restatement's map: insert() runs insertScan on a cloud of 16-byte points from an origin."""

    def __init__(self, **params):
        p = dict(DEFAULTS)
        p.update(params)
        self._L = _lib("octomap_literal.cpp")
        self.resolution = p["resolution"]
        self._h = self._L.oct_new(self.resolution)
        self.set_params(**{k: v for k, v in p.items() if k != "resolution"})

    def set_params(self, **params):
        """Probabilities, clamps, threshold and max_range (the map is kept)."""
        p = dict(DEFAULTS)
        p.update(getattr(self, "_params", {}))
        p.update(params)
        self._params = {k: v for k, v in p.items() if k != "resolution"}
        self._L.oct_set_params(self._h, p["prob_hit"], p["prob_miss"], p["clamp_min"], p["clamp_max"],
                               p["occupancy_thres"], p["max_range"])

    def clear(self):
        self._L.oct_clear(self._h)

    def insert(self, cloud, origin=(0.0, 0.0, 0.0)):
        pts = np.ascontiguousarray(np.frombuffer(np.ascontiguousarray(cloud).tobytes(), np.float32).reshape(-1, 4))
        o = np.asarray(origin, np.float32)
        self._L.oct_insert(self._h, pts.ctypes.data_as(_FP), len(pts), float(o[0]), float(o[1]), float(o[2]))

    def voxels(self):
        """(keys (n, 3) uint16, log-odds float32) in leaf-iterator order."""
        n = self._L.oct_voxels(self._h, None, None, 0)
        keys, lo = np.empty(max(n, 1), np.uint64), np.empty(max(n, 1), np.float32)
        self._L.oct_voxels(self._h, keys.ctypes.data_as(_U64P), lo.ctypes.data_as(_FP), n)
        keys, lo = keys[:n], lo[:n]
        return np.stack([(keys >> np.uint64(16 * a)) & np.uint64(0xFFFF) for a in range(3)], 1).astype(np.uint16), lo

    def centers(self) -> np.ndarray:
        n = self._L.oct_centers(self._h, None, 0)
        out = np.empty((max(n, 1), 4), np.float32)
        self._L.oct_centers(self._h, out.ctypes.data_as(_FP), n)
        return out[:n]

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._L.oct_free(h)
            self._h = None
