"""disparity_to_point_cloud_b200 -- thin ctypes binding of libd2pc_b200.so.

The product is the C-ABI shared library (include/d2pc_b200.h) and the C++ host
mirror above it (csrc/node.hpp); this module only exists so that tests/ and
bench.py can drive the C ABI from Python.  It never computes anything itself
and never imports the CPU oracle: if the CUDA library is missing or no B200 is
present, every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libd2pc_b200.so")

FILTER_CROP, FILTER_CROP_FINITE, FILTER_VOXEL = 0, 1, 2
ARITH_EXACT, ARITH_FAST = 0, 1


class D2pcError(RuntimeError):
    def __init__(self, status: int, where: str, detail: str = ""):
        self.status = status
        msg = f"{where}: {_strerror(status)} ({status})"
        if detail:
            msg += f" [{detail}]"
        super().__init__(msg)


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double), ("baseline", C.c_double),
        ("rect_width", C.c_int32), ("rect_height", C.c_int32),
        ("border", C.c_int32), ("median_ksize", C.c_int32), ("disparity_scale", C.c_float),
        ("filter_mode", C.c_int32), ("arith_mode", C.c_int32),
        ("frame_id", C.c_char * 64), ("verbose", C.c_int32),
        ("offset_x", C.c_int32), ("offset_y", C.c_int32), ("fuse_rule", C.c_int32), ("fuse_median_ksize", C.c_int32),
        ("fuse_crop_left", C.c_int32), ("fuse_crop_right", C.c_int32), ("fuse_crop_top", C.c_int32),
        ("fuse_crop_bottom", C.c_int32),
        ("max_width", C.c_int32), ("max_height", C.c_int32), ("max_batch", C.c_int32), ("n_slots", C.c_int32),
    ]


class PointField(C.Structure):
    _fields_ = [("name", C.c_char * 8), ("offset", C.c_uint32), ("datatype", C.c_uint8), ("count", C.c_uint32)]


class Cloud(C.Structure):
    _fields_ = [
        ("data", C.POINTER(C.c_uint8)), ("height", C.c_uint32), ("width", C.c_uint32), ("point_step", C.c_uint32),
        ("row_step", C.c_uint32), ("is_bigendian", C.c_uint8), ("is_dense", C.c_uint8), ("n_fields", C.c_uint32),
        ("fields", PointField * 3),
    ]

    def bytes_view(self) -> np.ndarray:
        n = self.row_step * self.height
        if n == 0:
            return np.empty(0, dtype=np.uint8)
        return np.ctypeslib.as_array(self.data, shape=(n,))


class VoxelGrid(C.Structure):
    """d2pc_voxel_grid: pcl::VoxelGrid<PointXYZ> parameters of D2PC_FILTER_VOXEL."""
    _fields_ = [("struct_size", C.c_uint32), ("leaf_x", C.c_float), ("leaf_y", C.c_float), ("leaf_z", C.c_float),
                ("min_points_per_voxel", C.c_uint32), ("limit_field", C.c_int32), ("limit_min", C.c_double),
                ("limit_max", C.c_double)]


class RadiusOutlier(C.Structure):
    """d2pc_radius_outlier: pcl::RadiusOutlierRemoval parameters of the stage behind every filter mode."""
    _fields_ = [("struct_size", C.c_uint32), ("radius", C.c_double), ("min_neighbors", C.c_uint32)]


class CropBox(C.Structure):
    """d2pc_crop_box: pcl::CropBox (setTransform) parameters of the stage in front of VOXEL and the outlier stage."""
    _fields_ = [("struct_size", C.c_uint32), ("enabled", C.c_int32), ("min_pt", C.c_float * 3),
                ("max_pt", C.c_float * 3), ("transform", C.c_float * 12)]


class CloudTransform(C.Structure):
    """d2pc_cloud_transform: pcl::transformPointCloud matrix of the first cloud stage (camera frame -> target frame)."""
    _fields_ = [("struct_size", C.c_uint32), ("enabled", C.c_int32), ("matrix", C.c_float * 12)]


class LaserScanParams(C.Structure):
    """d2pc_laser_scan_params: pointcloud_to_laserscan's parameters of the scan output (and keep_cloud)."""
    _fields_ = [("struct_size", C.c_uint32), ("enabled", C.c_int32), ("min_height", C.c_double),
                ("max_height", C.c_double), ("angle_min", C.c_double), ("angle_max", C.c_double),
                ("angle_increment", C.c_double), ("scan_time", C.c_double), ("range_min", C.c_double),
                ("range_max", C.c_double), ("use_inf", C.c_int32), ("inf_epsilon", C.c_double),
                ("keep_cloud", C.c_int32)]


class OccupancyParams(C.Structure):
    """d2pc_occupancy_params: octomap_server's parameters of the occupancy map (and keep_cloud)."""
    _fields_ = [("struct_size", C.c_uint32), ("enabled", C.c_int32), ("resolution", C.c_double),
                ("prob_hit", C.c_double), ("prob_miss", C.c_double), ("clamp_min", C.c_double),
                ("clamp_max", C.c_double), ("occupancy_thres", C.c_double), ("max_range", C.c_double),
                ("max_bricks", C.c_uint32), ("keep_cloud", C.c_int32)]


class OccupancyInfo(C.Structure):
    """d2pc_occupancy_info: the map's counters (d2pc_occupancy_stats)."""
    _fields_ = [("frames_inserted", C.c_uint64), ("frames_dropped", C.c_uint64), ("known_voxels", C.c_uint64),
                ("occupied_voxels", C.c_uint64), ("bricks_used", C.c_uint64), ("bricks_capacity", C.c_uint64)]

    def as_dict(self) -> dict:
        return {f[0]: int(getattr(self, f[0])) for f in self._fields_}


class Octomap(C.Structure):
    """d2pc_octomap: octomap_msgs/Octomap data in library-owned memory."""
    _fields_ = [("data", C.POINTER(C.c_uint8)), ("size", C.c_uint64), ("resolution", C.c_double),
                ("binary", C.c_int32)]


class ProjectedMapParams(C.Structure):
    """d2pc_projected_map_params: octomap_server's parameters of the projected 2-D map."""
    _fields_ = [("struct_size", C.c_uint32), ("occupancy_min_z", C.c_double), ("occupancy_max_z", C.c_double),
                ("min_x_size", C.c_double), ("min_y_size", C.c_double)]


class GridMap(C.Structure):
    """d2pc_grid_map: nav_msgs/OccupancyGrid's info and its cells in library-owned memory."""
    _fields_ = [("data", C.POINTER(C.c_int8)), ("width", C.c_uint32), ("height", C.c_uint32),
                ("resolution", C.c_float), ("origin_x", C.c_double), ("origin_y", C.c_double)]


class LaserScan(C.Structure):
    """d2pc_laser_scan: the message fields of a scan and its library-owned ranges."""
    _fields_ = [("angle_min", C.c_float), ("angle_max", C.c_float), ("angle_increment", C.c_float),
                ("time_increment", C.c_float), ("scan_time", C.c_float), ("range_min", C.c_float),
                ("range_max", C.c_float), ("n_ranges", C.c_uint32), ("ranges", C.POINTER(C.c_float))]

    FIELDS = ("angle_min", "angle_max", "angle_increment", "time_increment", "scan_time", "range_min", "range_max")

    def fields(self) -> dict:
        return {k: getattr(self, k) for k in self.FIELDS}

    def ranges_array(self) -> np.ndarray:
        """A copy of the ranges (float32)."""
        if self.n_ranges == 0:
            return np.empty(0, np.float32)
        return np.ctypeslib.as_array(self.ranges, shape=(self.n_ranges,)).copy()


class Timing(C.Structure):
    _fields_ = [("h2d_us", C.c_float), ("kernels_us", C.c_float), ("d2h_us", C.c_float), ("total_us", C.c_float),
                ("points", C.c_uint64)]


class Image(C.Structure):
    _fields_ = [("data", C.POINTER(C.c_uint8)), ("width", C.c_uint32), ("height", C.c_uint32), ("step", C.c_uint32)]

    def array(self) -> np.ndarray:
        a = np.ctypeslib.as_array(self.data, shape=(self.height, self.step))
        return a[:, : self.width]


CLOUD_SINK = C.CFUNCTYPE(None, C.c_void_p, C.c_uint64, C.POINTER(Cloud))

# every symbol include/d2pc_b200.h declares: (name, restype, argtypes)
_u8p, _f32p, _f64p, _i32p, _u32p = (C.POINTER(t) for t in (C.c_uint8, C.c_float, C.c_double, C.c_int, C.c_uint32))
_ctx = C.c_void_p
SYMBOLS = [
    ("d2pc_config_default", None, [C.POINTER(Config)]),
    ("d2pc_create", C.c_int, [C.POINTER(Config), C.c_int, C.POINTER(_ctx)]),
    ("d2pc_destroy", None, [_ctx]),
    ("d2pc_q_from_intrinsics", C.c_int, [C.c_double] * 5 + [C.c_int, C.c_int, _f64p]),
    ("d2pc_set_q", C.c_int, [_ctx, _f64p]),
    ("d2pc_get_q", C.c_int, [_ctx, _f64p]),
    ("d2pc_set_filter_mode", C.c_int, [_ctx, C.c_int]),
    ("d2pc_set_arith_mode", C.c_int, [_ctx, C.c_int]),
    ("d2pc_voxel_grid_default", None, [C.POINTER(VoxelGrid)]),
    ("d2pc_set_voxel_grid", C.c_int, [_ctx, C.POINTER(VoxelGrid)]),
    ("d2pc_get_voxel_grid", C.c_int, [_ctx, C.POINTER(VoxelGrid)]),
    ("d2pc_radius_outlier_default", None, [C.POINTER(RadiusOutlier)]),
    ("d2pc_set_radius_outlier", C.c_int, [_ctx, C.POINTER(RadiusOutlier)]),
    ("d2pc_get_radius_outlier", C.c_int, [_ctx, C.POINTER(RadiusOutlier)]),
    ("d2pc_radius_outlier_device", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t, C.c_void_p,
                                             C.c_void_p, C.c_size_t, C.c_void_p]),
    ("d2pc_crop_box_default", None, [C.POINTER(CropBox)]),
    ("d2pc_set_crop_box", C.c_int, [_ctx, C.POINTER(CropBox)]),
    ("d2pc_get_crop_box", C.c_int, [_ctx, C.POINTER(CropBox)]),
    ("d2pc_crop_box_device", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t, C.c_void_p,
                                       C.c_void_p, C.c_size_t, C.c_void_p]),
    ("d2pc_cloud_transform_default", None, [C.POINTER(CloudTransform)]),
    ("d2pc_set_cloud_transform", C.c_int, [_ctx, C.POINTER(CloudTransform)]),
    ("d2pc_get_cloud_transform", C.c_int, [_ctx, C.POINTER(CloudTransform)]),
    ("d2pc_cloud_transform_device", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t, C.c_void_p,
                                              C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    ("d2pc_laser_scan_params_default", None, [C.POINTER(LaserScanParams)]),
    ("d2pc_set_laser_scan", C.c_int, [_ctx, C.POINTER(LaserScanParams)]),
    ("d2pc_get_laser_scan", C.c_int, [_ctx, C.POINTER(LaserScanParams)]),
    ("d2pc_laser_scan_ranges", C.c_int, [C.POINTER(LaserScanParams), _u32p]),
    ("d2pc_last_scan", C.c_int, [_ctx, C.POINTER(LaserScan)]),
    ("d2pc_laser_scan_device", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t, C.c_void_p,
                                         C.c_void_p, C.c_size_t]),
    ("d2pc_occupancy_params_default", None, [C.POINTER(OccupancyParams)]),
    ("d2pc_set_occupancy", C.c_int, [_ctx, C.POINTER(OccupancyParams)]),
    ("d2pc_get_occupancy", C.c_int, [_ctx, C.POINTER(OccupancyParams)]),
    ("d2pc_occupancy_reset", C.c_int, [_ctx]),
    ("d2pc_occupancy_stats", C.c_int, [_ctx, C.POINTER(OccupancyInfo)]),
    ("d2pc_occupancy_centers", C.c_int, [_ctx, C.c_void_p, C.c_size_t, C.POINTER(Cloud)]),
    ("d2pc_occupancy_voxels", C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    ("d2pc_occupancy_insert_device", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t, C.c_void_p,
                                               C.c_void_p]),
    ("d2pc_occupancy_octomap", C.c_int, [_ctx, C.c_int, C.POINTER(Octomap)]),
    ("d2pc_projected_map_params_default", None, [C.POINTER(ProjectedMapParams)]),
    ("d2pc_occupancy_projected_map", C.c_int, [_ctx, C.POINTER(ProjectedMapParams), C.POINTER(GridMap)]),
    ("d2pc_process_mono8", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(Cloud)]),
    ("d2pc_process_f32", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(Cloud)]),
    ("d2pc_submit_mono8", C.c_int, [_ctx, C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    ("d2pc_submit_f32", C.c_int, [_ctx, C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    ("d2pc_wait", C.c_int, [_ctx, C.c_int, C.POINTER(Cloud)]),
    ("d2pc_submit_mono8_into", C.c_int, [_ctx, C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                         C.c_size_t]),
    ("d2pc_submit_f32_into", C.c_int, [_ctx, C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                       C.c_size_t]),
    ("d2pc_process_mono8_into", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t,
                                          C.POINTER(Cloud)]),
    ("d2pc_process_f32_into", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t,
                                        C.POINTER(Cloud)]),
    ("d2pc_set_timing", C.c_int, [_ctx, C.c_int]),
    ("d2pc_slot_timing", C.c_int, [_ctx, C.c_int, C.POINTER(Timing)]),
    ("d2pc_host_alloc", C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    ("d2pc_host_free", C.c_int, [C.c_void_p]),
    ("d2pc_host_register", C.c_int, [C.c_void_p, C.c_size_t]),
    ("d2pc_host_unregister", C.c_int, [C.c_void_p]),
    ("d2pc_process_stream", C.c_int, [_ctx, C.c_void_p, C.c_uint64, C.c_size_t, C.c_uint64, C.c_int, C.c_uint32,
                                      C.c_uint32, C.c_uint32, CLOUD_SINK, C.c_void_p]),
    ("d2pc_reproject_f32_device", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_size_t,
                                            C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    ("d2pc_reproject_mono8_device", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_size_t,
                                              C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    ("d2pc_median_u8_device", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t, C.c_void_p,
                                        C.c_size_t, C.c_int]),
    ("d2pc_compute_stream", C.c_void_p, [_ctx]),
    ("d2pc_sync", C.c_int, [_ctx]),
    ("d2pc_launch_count", C.c_uint64, [_ctx]),
    ("d2pc_fuse_geometry", C.c_int, [_ctx, C.c_uint32, C.c_uint32, _i32p, _i32p, _i32p, _i32p]),
    ("d2pc_fuse", C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                            C.c_uint32, C.POINTER(Image), C.POINTER(Image)]),
    ("d2pc_preprocess_score", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int,
                                        C.POINTER(Image)]),
    ("d2pc_preprocess_score_device", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t, C.c_int,
                                               C.c_void_p]),
    ("d2pc_fuse_preprocessed", C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                         C.c_uint32, C.POINTER(Image), C.POINTER(Image)]),
    ("d2pc_colorize_depth", C.c_int, [_ctx, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(Image)]),
    ("d2pc_fuse_device", C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                   C.c_size_t, C.c_void_p, C.c_void_p]),
    ("d2pc_fuse_preprocessed_device", C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                                C.c_uint32, C.c_size_t, C.c_void_p, C.c_void_p]),
    ("d2pc_fuse_then_process", C.c_int, [_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                         C.c_uint32, C.c_uint32, C.POINTER(Cloud)]),
    ("d2pc_submit_fusion", C.c_int, [_ctx, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                     C.c_uint32, C.c_uint32, C.c_int]),
    ("d2pc_process_fusion_stream", C.c_int, [_ctx, C.c_void_p, C.c_uint64, C.c_size_t, C.c_uint64, C.c_uint32,
                                             C.c_uint32, C.c_uint32, C.c_int, CLOUD_SINK, C.c_void_p]),
    ("d2pc_serialize_pointcloud2", C.c_size_t, [_ctx, C.POINTER(Cloud), C.c_uint32, C.c_uint32, C.c_uint32,
                                                C.c_void_p, C.c_size_t]),
    ("d2pc_serialize_laserscan", C.c_size_t, [_ctx, C.POINTER(LaserScan), C.c_uint32, C.c_uint32, C.c_uint32,
                                              C.c_void_p, C.c_size_t]),
    ("d2pc_set_tuning", C.c_int, [_ctx, C.c_char_p, C.c_int]),
    ("d2pc_strerror", C.c_char_p, [C.c_int]),
    ("d2pc_last_cuda_error", C.c_char_p, [_ctx]),
    ("d2pc_abi_version", C.c_int, []),
    ("d2pc_device_count", C.c_int, []),
]

_lib = None


def lib() -> C.CDLL:
    """Loads libd2pc_b200.so.  Raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(
                f"{LIB_PATH} is missing: build it with `python -m disparity_to_point_cloud_b200.build` "
                "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _strerror(status: int) -> str:
    try:
        return lib().d2pc_strerror(status).decode()
    except Exception:  # pragma: no cover
        return "?"


def default_config() -> Config:
    c = Config()
    lib().d2pc_config_default(C.byref(c))
    return c


def q_from_intrinsics(fx=714.24, fy=713.5, cx=376.0, cy=240.0, baseline=0.09, rect_w=752, rect_h=480) -> np.ndarray:
    q = np.zeros(16, dtype=np.float64)
    rc = lib().d2pc_q_from_intrinsics(fx, fy, cx, cy, baseline, rect_w, rect_h, q.ctypes.data_as(_f64p))
    if rc:
        raise D2pcError(rc, "d2pc_q_from_intrinsics")
    return q.reshape(4, 4)


def laser_scan_params(**params) -> LaserScanParams:
    """d2pc_laser_scan_params_default with `params` (any field of LaserScanParams) set on top; enabled defaults to 1."""
    p = LaserScanParams()
    lib().d2pc_laser_scan_params_default(C.byref(p))
    p.enabled = 1
    for k, v in params.items():
        if k not in {f[0] for f in LaserScanParams._fields_} or k == "struct_size":
            raise ValueError(f"laser_scan_params: unknown parameter {k!r}")
        setattr(p, k, v)
    return p


def occupancy_params(**params) -> OccupancyParams:
    """d2pc_occupancy_params_default with `params` (any field of OccupancyParams) set on top; enabled defaults to 1."""
    p = OccupancyParams()
    lib().d2pc_occupancy_params_default(C.byref(p))
    p.enabled = 1
    for k, v in params.items():
        if k not in {f[0] for f in OccupancyParams._fields_} or k == "struct_size":
            raise ValueError(f"occupancy_params: unknown parameter {k!r}")
        setattr(p, k, v)
    return p


def laser_scan_ranges(**params) -> int:
    """The number of ranges pointcloud_to_laserscan makes for these params (d2pc_laser_scan_ranges)."""
    n = C.c_uint32()
    rc = lib().d2pc_laser_scan_ranges(C.byref(laser_scan_params(**params)), C.byref(n))
    if rc:
        raise D2pcError(rc, "d2pc_laser_scan_ranges")
    return int(n.value)


class PinnedArray:
    """numpy view over cudaHostAlloc memory (d2pc_host_alloc)."""

    def __init__(self, shape, dtype):
        self.dtype = np.dtype(dtype)
        self.shape = tuple(shape)
        n = int(np.prod(self.shape)) * self.dtype.itemsize
        self._ptr = C.c_void_p()
        rc = lib().d2pc_host_alloc(C.byref(self._ptr), max(n, 1))
        if rc:
            raise D2pcError(rc, "d2pc_host_alloc")
        buf = (C.c_uint8 * max(n, 1)).from_address(self._ptr.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self._ptr:
            self.array = None
            lib().d2pc_host_free(self._ptr)
            self._ptr = None


class RegisteredArray:
    """Page-locks an existing numpy array in place (d2pc_host_register) for the lifetime of this object."""

    def __init__(self, array: np.ndarray):
        assert array.flags["C_CONTIGUOUS"]
        self.array = array
        rc = lib().d2pc_host_register(array.ctypes.data, array.nbytes)
        if rc:
            raise D2pcError(rc, "d2pc_host_register")
        self._live = True

    def free(self):
        if self._live:
            lib().d2pc_host_unregister(self.array.ctypes.data)
            self._live = False

    def __del__(self):  # pragma: no cover
        try:
            self.free()
        except Exception:
            pass


class Context:
    """One d2pc_ctx: the GPU stand-in for a Disparity2PCloud / DepthMapFusion node object."""

    def __init__(self, device: int = 0, config: Config | None = None, **overrides):
        cfg = config or default_config()
        for k, v in overrides.items():
            if k == "frame_id":
                v = v.encode() if isinstance(v, str) else v
            setattr(cfg, k, v)
        self.cfg = cfg
        self._h = _ctx()
        rc = lib().d2pc_create(C.byref(cfg), device, C.byref(self._h))
        if rc:
            raise D2pcError(rc, "d2pc_create")
        self._keep = {}

    # -- lifecycle
    def close(self):
        if self._h:
            lib().d2pc_destroy(self._h)
            self._h = None
        self._keep = {}

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, where):
        if rc:
            raise D2pcError(rc, where, lib().d2pc_last_cuda_error(self._h).decode())

    # -- parameters
    def set_q(self, q):
        q = np.ascontiguousarray(np.asarray(q, dtype=np.float64).reshape(16))
        self._check(lib().d2pc_set_q(self._h, q.ctypes.data_as(_f64p)), "d2pc_set_q")

    def get_q(self) -> np.ndarray:
        q = np.zeros(16, dtype=np.float64)
        self._check(lib().d2pc_get_q(self._h, q.ctypes.data_as(_f64p)), "d2pc_get_q")
        return q.reshape(4, 4)

    def set_filter_mode(self, m):
        self._check(lib().d2pc_set_filter_mode(self._h, m), "d2pc_set_filter_mode")

    def set_voxel_grid(self, leaf, min_points: int = 0, limit=None):
        """pcl::VoxelGrid parameters for FILTER_VOXEL.  leaf: one size or (x, y, z); limit: None or
        (field, lo, hi) with field "x", "y" or "z" (both ends inclusive)."""
        g = VoxelGrid()
        lib().d2pc_voxel_grid_default(C.byref(g))
        lx, ly, lz = (leaf, leaf, leaf) if np.isscalar(leaf) else leaf
        g.leaf_x, g.leaf_y, g.leaf_z = lx, ly, lz
        g.min_points_per_voxel = int(min_points)
        if limit is not None:
            field, lo, hi = limit
            g.limit_field = {"x": 0, "y": 1, "z": 2}[field]
            g.limit_min, g.limit_max = float(lo), float(hi)
        self._check(lib().d2pc_set_voxel_grid(self._h, C.byref(g)), "d2pc_set_voxel_grid")

    def get_voxel_grid(self) -> VoxelGrid:
        g = VoxelGrid()
        self._check(lib().d2pc_get_voxel_grid(self._h, C.byref(g)), "d2pc_get_voxel_grid")
        return g

    def set_radius_outlier(self, radius: float, min_neighbors: int = 1):
        """pcl::RadiusOutlierRemoval behind the filter mode: radius 0 turns the stage off."""
        if not 0 <= int(min_neighbors) <= 0xFFFFFFFF:  # ctypes would wrap a negative count into a huge one
            raise ValueError(f"set_radius_outlier: min_neighbors must be in [0, 2^32 - 1], got {min_neighbors}")
        p = RadiusOutlier()
        lib().d2pc_radius_outlier_default(C.byref(p))
        p.radius = float(radius)
        p.min_neighbors = int(min_neighbors)
        self._check(lib().d2pc_set_radius_outlier(self._h, C.byref(p)), "d2pc_set_radius_outlier")

    def get_radius_outlier(self) -> RadiusOutlier:
        p = RadiusOutlier()
        self._check(lib().d2pc_get_radius_outlier(self._h, C.byref(p)), "d2pc_get_radius_outlier")
        return p

    @staticmethod
    def _affine(m, what) -> np.ndarray:
        """A 3x4 [A | t], or a 4x4 matrix whose last row is (0, 0, 0, 1), as 12 row-major float32 values."""
        t = np.asarray(m, np.float32)
        if t.shape == (4, 4):
            if not np.array_equal(t[3], np.float32([0, 0, 0, 1])):
                raise ValueError(f"{what}: the last row of a 4x4 transform must be (0, 0, 0, 1), got {t[3]}")
            t = t[:3]
        if t.shape != (3, 4):
            raise ValueError(f"{what}: transform must be 3x4 or 4x4, got {t.shape}")
        return t.reshape(12)

    def set_crop_box(self, min_pt, max_pt=None, transform=None):
        """pcl::CropBox in front of VOXEL and the outlier stage: keep the points p with min_pt <= T p <= max_pt.
        transform: None (the identity) or the camera -> box transform T as a 3x4 [R | t] or a 4x4 matrix whose last
        row is (0, 0, 0, 1).  set_crop_box(None) turns the box off."""
        b = CropBox()
        lib().d2pc_crop_box_default(C.byref(b))
        if min_pt is not None:
            if max_pt is None:
                raise ValueError("set_crop_box: max_pt is required with min_pt")
            b.enabled = 1
            b.min_pt[:] = [float(v) for v in np.asarray(min_pt, np.float32).reshape(3)]
            b.max_pt[:] = [float(v) for v in np.asarray(max_pt, np.float32).reshape(3)]
            if transform is not None:
                b.transform[:] = [float(v) for v in self._affine(transform, "set_crop_box")]
        self._check(lib().d2pc_set_crop_box(self._h, C.byref(b)), "d2pc_set_crop_box")

    def get_crop_box(self) -> CropBox:
        b = CropBox()
        self._check(lib().d2pc_get_crop_box(self._h, C.byref(b)), "d2pc_get_crop_box")
        return b

    def set_transform(self, matrix):
        """pcl::transformPointCloud as the first cloud stage: every finite point p becomes T p (camera frame ->
        target frame), in front of the crop box, VOXEL and the outlier stage.  matrix: a 3x4 [A | t] or a 4x4 matrix
        whose last row is (0, 0, 0, 1); None turns the transform off.  A slot uses the setting in force when its frame
        is submitted."""
        t = CloudTransform()
        lib().d2pc_cloud_transform_default(C.byref(t))
        if matrix is not None:
            t.enabled = 1
            t.matrix[:] = [float(v) for v in self._affine(matrix, "set_transform")]
        self._check(lib().d2pc_set_cloud_transform(self._h, C.byref(t)), "d2pc_set_cloud_transform")

    def get_transform(self) -> CloudTransform:
        t = CloudTransform()
        self._check(lib().d2pc_get_cloud_transform(self._h, C.byref(t)), "d2pc_get_cloud_transform")
        return t

    def set_laser_scan(self, enabled: bool = True, **params):
        """pointcloud_to_laserscan as an output next to the cloud: the scan of every cloud a host entry publishes,
        read with last_scan().  params: any field of LaserScanParams (the nodelet's ten params and keep_cloud);
        set_laser_scan(False) turns it off."""
        p = laser_scan_params(**params)
        p.enabled = 1 if enabled else 0
        self._check(lib().d2pc_set_laser_scan(self._h, C.byref(p)), "d2pc_set_laser_scan")

    def get_laser_scan(self) -> LaserScanParams:
        p = LaserScanParams()
        self._check(lib().d2pc_get_laser_scan(self._h, C.byref(p)), "d2pc_get_laser_scan")
        return p

    def last_scan_raw(self) -> LaserScan:
        """d2pc_last_scan as it is (its ranges point into library memory)."""
        s = LaserScan()
        self._check(lib().d2pc_last_scan(self._h, C.byref(s)), "d2pc_last_scan")
        return s

    def last_scan(self):
        """The scan of the cloud last returned: (dict of the seven float fields, float32 ranges)."""
        s = self.last_scan_raw()
        return s.fields(), s.ranges_array()

    def laser_scan_device(self, d_in, n_frames, n_max, in_stride, d_in_counts, d_ranges, ranges_stride):
        """d2pc_laser_scan_device: the context's (enabled) scan of clouds on the device, frame f's ranges at
        d_ranges + f * ranges_stride bytes."""
        self._check(lib().d2pc_laser_scan_device(self._h, d_in, n_frames, n_max, in_stride, d_in_counts or None,
                                                 d_ranges, ranges_stride), "d2pc_laser_scan_device")

    def serialize_laserscan(self, scan: LaserScan, seq=0, sec=0, nsec=0) -> bytes:
        need = lib().d2pc_serialize_laserscan(self._h, C.byref(scan), seq, sec, nsec, None, 0)
        buf = (C.c_uint8 * need)()
        lib().d2pc_serialize_laserscan(self._h, C.byref(scan), seq, sec, nsec, buf, need)
        return bytes(buf)

    def set_occupancy(self, enabled: bool = True, **params):
        """octomap_server's insertScan as a map the context keeps on the device, updated by every cloud a host entry
        publishes.  params: any field of OccupancyParams; set_occupancy(False) stops updates and keeps the map."""
        p = occupancy_params(**params)
        p.enabled = 1 if enabled else 0
        self._check(lib().d2pc_set_occupancy(self._h, C.byref(p)), "d2pc_set_occupancy")

    def get_occupancy(self) -> OccupancyParams:
        p = OccupancyParams()
        self._check(lib().d2pc_get_occupancy(self._h, C.byref(p)), "d2pc_get_occupancy")
        return p

    def occupancy_reset(self):
        self._check(lib().d2pc_occupancy_reset(self._h), "d2pc_occupancy_reset")

    def occupancy_stats(self) -> dict:
        s = OccupancyInfo()
        self._check(lib().d2pc_occupancy_stats(self._h, C.byref(s)), "d2pc_occupancy_stats")
        return s.as_dict()

    def occupancy_centers(self) -> np.ndarray:
        """The centres of the occupied voxels in Morton order, an (n, 4) float32 array of PointXYZ {x, y, z, 1}."""
        cl = Cloud()
        rc = lib().d2pc_occupancy_centers(self._h, None, 0, C.byref(cl))
        if rc not in (0, -9):
            self._check(rc, "d2pc_occupancy_centers")
        while True:
            out = np.empty((max(int(cl.width), 1), 4), np.float32)
            rc = lib().d2pc_occupancy_centers(self._h, out.ctypes.data, out.nbytes, C.byref(cl))
            if rc != -9:  # the map may have grown in between (frames still in flight): size again
                break
        self._check(rc, "d2pc_occupancy_centers")
        return out[: cl.width]

    def occupancy_voxels(self):
        """Every known voxel in Morton order: keys as an (n, 3) uint16 array (kx, ky, kz) and float32 log-odds."""
        n = C.c_uint64()
        rc = lib().d2pc_occupancy_voxels(self._h, None, None, 0, C.byref(n))
        while True:
            if rc not in (0, -9):
                self._check(rc, "d2pc_occupancy_voxels")
            keys, lo = np.empty(max(n.value, 1), np.uint64), np.empty(max(n.value, 1), np.float32)
            rc = lib().d2pc_occupancy_voxels(self._h, keys.ctypes.data, lo.ctypes.data, keys.size, C.byref(n))
            if rc != -9:
                break
        self._check(rc, "d2pc_occupancy_voxels")
        keys, lo = keys[: n.value], lo[: n.value]
        k3 = np.stack([(keys >> np.uint64(16 * a)) & np.uint64(0xFFFF) for a in range(3)], axis=1).astype(np.uint16)
        return k3, lo

    def occupancy_octomap(self, binary: bool = False) -> bytes:
        """The map as octomap_msgs/Octomap data (octomap_server's /octomap_full, or /octomap_binary with binary)."""
        m = Octomap()
        self._check(lib().d2pc_occupancy_octomap(self._h, 1 if binary else 0, C.byref(m)), "d2pc_occupancy_octomap")
        return C.string_at(m.data, m.size) if m.size else b""

    def occupancy_projected_map(self, occupancy_min_z: float = -sys.float_info.max,
                                occupancy_max_z: float = sys.float_info.max, min_x_size: float = 0.0,
                                min_y_size: float = 0.0):
        """The map projected to 2-D (octomap_server's /projected_map): (cells, resolution, (origin_x, origin_y)) with
        cells a (height, width) int8 copy of -1 / 0 / 100, row y, column x; (0, 0) for an empty map."""
        p = ProjectedMapParams()
        lib().d2pc_projected_map_params_default(C.byref(p))
        p.occupancy_min_z, p.occupancy_max_z = occupancy_min_z, occupancy_max_z
        p.min_x_size, p.min_y_size = min_x_size, min_y_size
        g = GridMap()
        self._check(lib().d2pc_occupancy_projected_map(self._h, C.byref(p), C.byref(g)), "d2pc_occupancy_projected_map")
        n = g.width * g.height
        cells = (np.ctypeslib.as_array(g.data, (n,)).copy() if n else np.zeros(0, np.int8)).reshape(g.height, g.width)
        return cells, float(g.resolution), (float(g.origin_x), float(g.origin_y))

    def occupancy_insert_device(self, d_in, n_frames, n_max, in_stride, d_in_counts, origins):
        """d2pc_occupancy_insert_device: clouds on the device into the map, frame f from origins[f] (host, (n, 3))."""
        o = np.ascontiguousarray(origins, np.float32).reshape(-1)
        assert o.size >= 3 * n_frames
        self._check(lib().d2pc_occupancy_insert_device(self._h, d_in, n_frames, n_max, in_stride, d_in_counts or None,
                                                       o.ctypes.data), "d2pc_occupancy_insert_device")

    def set_arith_mode(self, m):
        self._check(lib().d2pc_set_arith_mode(self._h, m), "d2pc_set_arith_mode")

    def set_timing(self, enable: bool = True):
        self._check(lib().d2pc_set_timing(self._h, 1 if enable else 0), "d2pc_set_timing")

    def slot_timing(self, slot: int = 0) -> Timing:
        t = Timing()
        self._check(lib().d2pc_slot_timing(self._h, slot, C.byref(t)), "d2pc_slot_timing")
        return t

    def set_tuning(self, key: str, value: int):
        self._check(lib().d2pc_set_tuning(self._h, key.encode(), int(value)), f"d2pc_set_tuning({key})")

    # -- host entry points (what DisparityCb does)
    @staticmethod
    def _frame(img, dtype):
        a = np.asarray(img)
        # a row stride the C ABI cannot express (negative, or smaller than a row) is repacked, not passed on
        if (a.dtype != dtype or a.ndim != 2 or a.strides[1] != a.itemsize or a.strides[0] < a.shape[1] * a.itemsize
                or a.strides[0] > 0xFFFFFFFF):
            a = np.ascontiguousarray(a, dtype=dtype)
        return a

    def process_into(self, frame, dst: np.ndarray) -> np.ndarray:
        """DisparityCb with a caller-supplied destination (d2pc_process_*_into): the cloud bytes land in `dst`
        (uint8, contiguous; DMA'd in place when it is PinnedArray / registered memory).  Returns dst[:n_bytes]."""
        a = self._frame(frame, np.float32 if np.asarray(frame).dtype == np.float32 else np.uint8)
        assert dst.dtype == np.uint8 and dst.flags["C_CONTIGUOUS"]
        cl = Cloud()
        fn = lib().d2pc_process_f32_into if a.dtype == np.float32 else lib().d2pc_process_mono8_into
        self._check(fn(self._h, a.ctypes.data, a.shape[1], a.shape[0], a.strides[0], dst.ctypes.data, dst.size,
                       C.byref(cl)), "d2pc_process_into")
        self.last_cloud = cl
        return dst.reshape(-1)[: cl.row_step * cl.height]

    def process_mono8(self, img, copy: bool = True) -> np.ndarray:
        """copy=False returns a view of the library-owned pinned buffer (valid until the next call)."""
        a = self._frame(img, np.uint8)
        cl = Cloud()
        self._check(lib().d2pc_process_mono8(self._h, a.ctypes.data, a.shape[1], a.shape[0], a.strides[0],
                                             C.byref(cl)), "d2pc_process_mono8")
        self.last_cloud = cl
        return cl.bytes_view().copy() if copy else cl.bytes_view()

    def process_f32(self, disp, copy: bool = True) -> np.ndarray:
        a = self._frame(disp, np.float32)
        cl = Cloud()
        self._check(lib().d2pc_process_f32(self._h, a.ctypes.data, a.shape[1], a.shape[0], a.strides[0],
                                           C.byref(cl)), "d2pc_process_f32")
        self.last_cloud = cl
        return cl.bytes_view().copy() if copy else cl.bytes_view()

    def submit(self, slot: int, frame, dst: np.ndarray | None = None):
        a = np.asarray(frame)
        assert a.ndim == 2 and a.strides[1] == a.itemsize and a.strides[0] >= a.shape[1] * a.itemsize
        self._keep[slot] = (a, dst)  # the frame (and destination) of a slot stay alive until it is waited on
        if dst is not None:
            assert dst.dtype == np.uint8 and dst.flags["C_CONTIGUOUS"] and a.dtype in (np.float32, np.uint8)
            fn = lib().d2pc_submit_f32_into if a.dtype == np.float32 else lib().d2pc_submit_mono8_into
            self._check(fn(self._h, slot, a.ctypes.data, a.shape[1], a.shape[0], a.strides[0], dst.ctypes.data,
                           dst.size), "d2pc_submit_into")
            return
        if a.dtype == np.float32:
            rc = lib().d2pc_submit_f32(self._h, slot, a.ctypes.data, a.shape[1], a.shape[0], a.strides[0])
        elif a.dtype == np.uint8:
            rc = lib().d2pc_submit_mono8(self._h, slot, a.ctypes.data, a.shape[1], a.shape[0], a.strides[0])
        else:
            raise D2pcError(-2, "submit")
        self._check(rc, "d2pc_submit")

    def wait(self, slot: int) -> np.ndarray:
        cl = Cloud()
        try:
            self._check(lib().d2pc_wait(self._h, slot, C.byref(cl)), "d2pc_wait")
        finally:
            kept = self._keep.pop(slot, None)
        self.last_cloud = cl
        if kept is not None and kept[1] is not None:
            return kept[1].reshape(-1)[: cl.row_step * cl.height]  # the caller's own buffer
        return cl.bytes_view().copy()

    def process_stream(self, frames: np.ndarray, collect: bool = True, sink=None, n_frames: int | None = None):
        """frames: (F,H,W) u8 or f32 (numpy or PinnedArray.array).  n_frames > F cycles through the array
        as a ring.  Returns the list of clouds if collect."""
        assert frames.ndim == 3 and frames.strides[2] == frames.itemsize
        out = []

        def _sink(user, idx, cloud):
            if sink is not None:
                sink(idx, cloud.contents)
            if collect:
                out.append(cloud.contents.bytes_view().copy())

        cb = CLOUD_SINK(_sink) if (collect or sink is not None) else C.cast(None, CLOUD_SINK)
        f, h, w = frames.shape
        rc = lib().d2pc_process_stream(self._h, frames.ctypes.data, n_frames or f, frames.strides[0], f,
                                       1 if frames.dtype == np.float32 else 0, w, h, frames.strides[1], cb, None)
        self._check(rc, "d2pc_process_stream")
        return out

    # -- device entry points (pointers are raw CUDA device addresses, e.g. torch.Tensor.data_ptr())
    def reproject_f32_device(self, d_disp, n_frames, w, h, step, frame_stride, d_points, points_stride, d_counts=0):
        self._check(lib().d2pc_reproject_f32_device(self._h, d_disp, n_frames, w, h, step, frame_stride, d_points,
                                                    points_stride, d_counts or None), "d2pc_reproject_f32_device")

    def reproject_mono8_device(self, d_img, n_frames, w, h, step, frame_stride, d_points, points_stride, d_counts=0):
        self._check(lib().d2pc_reproject_mono8_device(self._h, d_img, n_frames, w, h, step, frame_stride, d_points,
                                                      points_stride, d_counts or None), "d2pc_reproject_mono8_device")

    def radius_outlier_device(self, d_in, n_frames, n_max, in_stride, d_in_counts, d_out, out_stride, d_out_counts):
        self._check(lib().d2pc_radius_outlier_device(self._h, d_in, n_frames, n_max, in_stride, d_in_counts or None,
                                                     d_out, out_stride, d_out_counts or None),
                    "d2pc_radius_outlier_device")

    def crop_box_device(self, d_in, n_frames, n_max, in_stride, d_in_counts, d_out, out_stride, d_out_counts):
        self._check(lib().d2pc_crop_box_device(self._h, d_in, n_frames, n_max, in_stride, d_in_counts or None,
                                               d_out, out_stride, d_out_counts or None), "d2pc_crop_box_device")

    def transform_device(self, d_in, n_frames, n_max, in_stride, d_in_counts, d_out, out_stride, d_out_counts=0,
                         d_transforms=None):
        """d2pc_cloud_transform_device: d_transforms None applies the context's (enabled) setting, otherwise it is
        the device address of n_frames row-major 3x4 float32 matrices.  d_out may be d_in (same stride)."""
        self._check(lib().d2pc_cloud_transform_device(self._h, d_in, n_frames, n_max, in_stride, d_in_counts or None,
                                                      d_out, out_stride, d_out_counts or None, d_transforms or None),
                    "d2pc_cloud_transform_device")

    def median_u8_device(self, d_src, w, h, src_step, d_dst, dst_step, ksize):
        self._check(lib().d2pc_median_u8_device(self._h, d_src, w, h, src_step, d_dst, dst_step, ksize),
                    "d2pc_median_u8_device")

    def compute_stream(self) -> int:
        return int(lib().d2pc_compute_stream(self._h) or 0)

    def sync(self):
        self._check(lib().d2pc_sync(self._h), "d2pc_sync")

    def launch_count(self) -> int:
        return int(lib().d2pc_launch_count(self._h))

    # -- fusion
    def fuse_geometry(self, w, h):
        r1, r2, rc_, dims = (np.zeros(4, np.int32), np.zeros(4, np.int32), np.zeros(4, np.int32), np.zeros(3, np.int32))
        st = lib().d2pc_fuse_geometry(self._h, w, h, *(a.ctypes.data_as(_i32p) for a in (r1, r2, rc_, dims)))
        return st, tuple(map(int, r1)), tuple(map(int, r2)), tuple(map(int, rc_)), tuple(map(int, dims))

    @staticmethod
    def _same_shape(arrs, what):
        if any(a.ndim != 2 or a.shape != arrs[0].shape for a in arrs):
            raise ValueError(f"{what}: the input images must share one (H, W) shape, got {[a.shape for a in arrs]}")

    def fuse(self, d1, d2, s1, s2):
        arrs = [np.ascontiguousarray(a, dtype=np.uint8) for a in (d1, d2, s1, s2)]
        self._same_shape(arrs, "fuse")
        h, w = arrs[0].shape
        fused, combined = Image(), Image()
        self._check(lib().d2pc_fuse(self._h, *(a.ctypes.data for a in arrs), w, h, w, C.byref(fused),
                                    C.byref(combined)), "d2pc_fuse")
        return fused.array().copy(), combined.array().copy()

    def preprocess_score(self, score, which: int) -> np.ndarray:
        a = np.ascontiguousarray(score, dtype=np.uint8)
        h, w = a.shape
        out = Image()
        self._check(lib().d2pc_preprocess_score(self._h, a.ctypes.data, w, h, w, which, C.byref(out)),
                    "d2pc_preprocess_score")
        return out.array().copy()

    def preprocess_score_device(self, d_score, w, h, step, which, d_out):
        self._check(lib().d2pc_preprocess_score_device(self._h, d_score, w, h, step, which, d_out),
                    "d2pc_preprocess_score_device")

    def fuse_preprocessed(self, d1, d2, s1c, s2c):
        d1, d2 = (np.ascontiguousarray(a, dtype=np.uint8) for a in (d1, d2))
        s1c, s2c = (np.ascontiguousarray(a, dtype=np.uint8) for a in (s1c, s2c))
        self._same_shape([d1, d2], "fuse_preprocessed")
        h, w = d1.shape
        n = self.fuse_geometry(w, h)[4][0]
        if s1c.shape != (n, n) or s2c.shape != (n, n):
            raise ValueError(f"fuse_preprocessed: the score caches must be {n} x {n}, got {s1c.shape} and {s2c.shape}")
        fused, combined = Image(), Image()
        self._check(lib().d2pc_fuse_preprocessed(self._h, d1.ctypes.data, d2.ctypes.data, s1c.ctypes.data,
                                                 s2c.ctypes.data, w, h, w, C.byref(fused), C.byref(combined)),
                    "d2pc_fuse_preprocessed")
        return fused.array().copy(), combined.array().copy()

    def colorize_depth(self, gray) -> np.ndarray:
        a = np.ascontiguousarray(gray, dtype=np.uint8)
        h, w = a.shape
        out = Image()
        self._check(lib().d2pc_colorize_depth(self._h, a.ctypes.data, w, h, w, C.byref(out)), "d2pc_colorize_depth")
        return np.ctypeslib.as_array(out.data, shape=(h, 3 * w)).reshape(h, w, 3).copy()

    def fuse_device(self, d_d1, d_d2, d_s1, d_s2, w, h, step, d_fused, d_combined=0):
        self._check(lib().d2pc_fuse_device(self._h, d_d1, d_d2, d_s1, d_s2, w, h, step, d_fused, d_combined or None),
                    "d2pc_fuse_device")

    def fuse_preprocessed_device(self, d_d1, d_d2, d_s1c, d_s2c, w, h, step, d_fused, d_combined=0):
        self._check(lib().d2pc_fuse_preprocessed_device(self._h, d_d1, d_d2, d_s1c, d_s2c, w, h, step, d_fused,
                                                        d_combined or None), "d2pc_fuse_preprocessed_device")

    def fuse_then_process(self, d1, d2, s1, s2) -> np.ndarray:
        arrs = [np.ascontiguousarray(a, dtype=np.uint8) for a in (d1, d2, s1, s2)]
        self._same_shape(arrs, "fuse_then_process")
        h, w = arrs[0].shape
        cl = Cloud()
        self._check(lib().d2pc_fuse_then_process(self._h, *(a.ctypes.data for a in arrs), w, h, w, C.byref(cl)),
                    "d2pc_fuse_then_process")
        self.last_cloud = cl
        return cl.bytes_view().copy()

    def submit_fusion(self, slot: int, d1, d2, s1, s2, preprocess_scores: bool = True):
        """One whole fusion-node pass + DisparityCb on pipeline slot `slot` (collect with wait(slot))."""
        arrs = [np.asarray(a) for a in (d1, d2, s1, s2)]
        self._same_shape(arrs, "submit_fusion")
        assert all(a.dtype == np.uint8 and a.strides[1] == 1 and a.strides[0] == arrs[0].strides[0] for a in arrs)
        h, w = arrs[0].shape
        self._keep[slot] = (arrs, None)
        self._check(lib().d2pc_submit_fusion(self._h, slot, *(a.ctypes.data for a in arrs), w, h, arrs[0].strides[0],
                                             1 if preprocess_scores else 0), "d2pc_submit_fusion")

    def process_fusion_stream(self, sets: np.ndarray, preprocess_scores: bool = True, collect: bool = True, sink=None,
                              n_sets: int | None = None):
        """sets: (S, 4, H, W) uint8, the four frames of a set in the order d1, d2, s1, s2; n_sets > S cycles."""
        assert sets.ndim == 4 and sets.shape[1] == 4 and sets.dtype == np.uint8 and sets.strides[3] == 1
        assert sets.strides[1] == sets.strides[2] * sets.shape[2]
        out = []

        def _sink(user, idx, cloud):
            if sink is not None:
                sink(idx, cloud.contents)
            if collect:
                out.append(cloud.contents.bytes_view().copy())

        cb = CLOUD_SINK(_sink) if (collect or sink is not None) else C.cast(None, CLOUD_SINK)
        sn, _, h, w = sets.shape
        rc = lib().d2pc_process_fusion_stream(self._h, sets.ctypes.data, n_sets or sn, sets.strides[0], sn, w, h,
                                              sets.strides[2], 1 if preprocess_scores else 0, cb, None)
        self._check(rc, "d2pc_process_fusion_stream")
        return out

    def serialize_pointcloud2(self, cloud: Cloud, seq=0, sec=0, nsec=0) -> bytes:
        need = lib().d2pc_serialize_pointcloud2(self._h, C.byref(cloud), seq, sec, nsec, None, 0)
        buf = (C.c_uint8 * need)()
        lib().d2pc_serialize_pointcloud2(self._h, C.byref(cloud), seq, sec, nsec, buf, need)
        return bytes(buf)


def device_count() -> int:
    return int(lib().d2pc_device_count())
