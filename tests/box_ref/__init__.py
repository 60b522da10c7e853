"""ctypes view of the CPU references of the crop box stage (test infrastructure, not product code).

crop_box()  tests/box_ref/crop_box.c: the recipe of include/d2pc_b200.h.
pcl()       tests/box_ref/pcl_cropbox.cpp: CropBox::applyFilter's loop restated literally (identity shortcut,
            transformPoint order, rejection on < / >).

Both take a cloud of 16-byte points, the box's min_pt / max_pt and a 3x4 transform (None: the identity), and return
the PointCloud2.data bytes of the kept points (is_dense is always 1).  The sources are compiled on first use into a
per-user temporary directory keyed by their hash, so the repository tree is never written.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = {"crop_box.c": (["gcc", "-std=c11"], "d2pc_box_ref"), "pcl_cropbox.cpp": (["g++", "-std=c++14"],
                                                                                     "d2pc_box_pcl")}
_fns: dict[str, C._CFuncPtr] = {}
_FP = C.POINTER(C.c_float)
IDENTITY = np.eye(3, 4, dtype=np.float32)


def _fn(src: str):
    if src in _fns:
        return _fns[src]
    path = os.path.join(_HERE, src)
    digest = hashlib.sha256(open(path, "rb").read()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"d2pc_box_ref_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"{os.path.splitext(src)[0]}_{digest}.so")
    (compiler, std), name = _SOURCES[src]
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run([compiler, std, "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Werror", path,
                        "-o", tmp, "-lm"], check=True)
        os.replace(tmp, so)
    fn = getattr(C.CDLL(so), name)
    fn.argtypes = [_FP, C.c_size_t, _FP, _FP, _FP, _FP]
    fn.restype = C.c_size_t
    _fns[src] = fn
    return fn


def _f32(a, n) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, np.float32).reshape(n))


def _run(src: str, cloud, min_pt, max_pt, transform) -> bytes:
    pts = np.ascontiguousarray(np.frombuffer(np.ascontiguousarray(cloud).tobytes(), np.float32).reshape(-1, 4))
    mn, mx = _f32(min_pt, 3), _f32(max_pt, 3)
    t = _f32(IDENTITY if transform is None else transform, 12)
    out = np.empty(max(len(pts), 1) * 4, np.float32)
    k = _fn(src)(pts.ctypes.data_as(_FP), len(pts), mn.ctypes.data_as(_FP), mx.ctypes.data_as(_FP),
                 t.ctypes.data_as(_FP), out.ctypes.data_as(_FP))
    return out[: 4 * k].tobytes()


def crop_box(cloud, min_pt, max_pt, transform=None) -> bytes:
    return _run("crop_box.c", cloud, min_pt, max_pt, transform)


def pcl(cloud, min_pt, max_pt, transform=None) -> bytes:
    return _run("pcl_cropbox.cpp", cloud, min_pt, max_pt, transform)
