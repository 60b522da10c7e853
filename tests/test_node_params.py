"""CPU: the point cloud node's params (include/d2pc_b200/node_params.hpp, read_cloud_settings) through the offline
harness's node1settings mode: every launch param lands in its settings field, an empty launch file gives the library's
d2pc_*_default values and the node's own defaults, and both bindings (the node mirror and the ROS1 shim) read their
params through that one reader."""
import ctypes as C
import glob
import math
import os
import subprocess

import numpy as np
import pytest

import disparity_to_point_cloud_b200 as d2pc
from conftest import ROOT

# param -> (launch value, settings field); every value differs from the field's default
PARAMS = {
    "fx_": ("700.5", "config.fx"), "fy_": ("701.25", "config.fy"), "cx_": ("370.5", "config.cx"),
    "cy_": ("230.25", "config.cy"), "base_line_": ("0.12", "config.baseline"),
    "voxel_z_min": ("-0.5", "voxel.limit_min"), "voxel_z_max": ("4.5", "voxel.limit_max"),
    "radius_outlier_radius": ("0.3", "ror_radius"), "radius_outlier_min_neighbors": ("4", "ror_min_neighbors"),
    "crop_box_enable": ("1", "crop_box.enabled"), "transform_enable": ("1", "transform.enabled"),
    "scan_enable": ("1", "scan.enabled"), "scan_min_height": ("0.1", "scan.min_height"),
    "scan_max_height": ("2.0", "scan.max_height"), "scan_angle_min": ("-1.0", "scan.angle_min"),
    "scan_angle_max": ("1.25", "scan.angle_max"), "scan_angle_increment": ("0.01", "scan.angle_increment"),
    "scan_scan_time": ("0.05", "scan.scan_time"), "scan_range_min": ("0.2", "scan.range_min"),
    "scan_range_max": ("20", "scan.range_max"), "scan_use_inf": ("0", "scan.use_inf"),
    "scan_inf_epsilon": ("0.5", "scan.inf_epsilon"), "scan_keep_cloud": ("0", "scan.keep_cloud"),
    "map_enable": ("1", "map.enabled"), "map_resolution": ("0.1", "map.resolution"),
    "map_sensor_model_hit": ("0.75", "map.prob_hit"), "map_sensor_model_miss": ("0.35", "map.prob_miss"),
    "map_sensor_model_min": ("0.15", "map.clamp_min"), "map_sensor_model_max": ("0.95", "map.clamp_max"),
    "map_occupancy_thres": ("0.6", "map.occupancy_thres"), "map_max_range": ("9.5", "map.max_range"),
    "map_max_bricks": ("5000", "map.max_bricks"), "map_keep_cloud": ("0", "map.keep_cloud"),
    "map_occupancy_min_z": ("-1.5", "projected_map.occupancy_min_z"),
    "map_occupancy_max_z": ("2.5", "projected_map.occupancy_max_z"),
    "map_min_x_size": ("10", "projected_map.min_x_size"), "map_min_y_size": ("12", "projected_map.min_y_size"),
}
LEAF = "0.07"  # voxel_leaf_size: all three leaf sizes, as float
BOX = {"min_x": "-2.5", "min_y": "-3.5", "min_z": "0.25", "max_x": "2.75", "max_y": "3.25", "max_z": "6.5"}
POSES = {"crop_box_": (0.5, -0.25, 1.5, 0.1, -0.2, 0.3), "transform_": (0.11, 0.22, 0.33, -0.4, 0.5, -0.6)}
POSE_NAMES = ("tx", "ty", "tz", "roll", "pitch", "yaw")


@pytest.fixture(scope="module")
def harness():
    from disparity_to_point_cloud_b200 import build
    build.build()
    return build.build_harness()


def settings(harness, tmp_path, params):
    launch = tmp_path / "n.launch"
    lines = "".join(f'    <param name="{k}" value="{v}"/>\n' for k, v in params.items())
    launch.write_text('<launch>\n  <node name="n" pkg="p" type="t">\n' + lines + "  </node>\n</launch>\n")
    out = subprocess.run([harness, "node1settings", str(launch)], check=True, capture_output=True, text=True).stdout
    got = dict(line.split(" ", 1) for line in out.splitlines())
    return {k: v if k == "frame_id" else float(v) for k, v in got.items()}


def pose_matrix(pose):
    """R = Rz(yaw) Ry(pitch) Rx(roll) next to t, row-major 3x4."""
    tx, ty, tz, r, p, y = pose
    cr, sr, cp, sp, cy, sy = math.cos(r), math.sin(r), math.cos(p), math.sin(p), math.cos(y), math.sin(y)
    return np.array([[cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr, tx],
                     [sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr, ty],
                     [-sp, cp * sr, cp * cr, tz]]).ravel()


def array(got, name, n):
    return np.array([got[f"{name}.{i}"] for i in range(n)])


def all_params():
    p = {k: v for k, (v, _) in PARAMS.items()}
    p["voxel_leaf_size"] = LEAF
    p.update({"crop_box_" + k: v for k, v in BOX.items()})
    for prefix, pose in POSES.items():
        p.update({prefix + n: repr(v) for n, v in zip(POSE_NAMES, pose)})
    p["transform_target_frame"] = "body"
    return p


def test_every_param_lands_in_its_field(harness, tmp_path):
    got = settings(harness, tmp_path, all_params())
    empty = settings(harness, tmp_path, {})
    for name, (value, field) in PARAMS.items():
        assert got[field] == float(value), (name, got[field])
        assert got[field] != empty[field], name  # the value is not the default
    assert got["voxel_on"] == 1 and got["voxel.limit_field"] == 2
    for a in "xyz":
        assert got[f"voxel.leaf_{a}"] == np.float32(LEAF)
    for i, a in enumerate("xyz"):
        assert got[f"crop_box.min_pt.{i}"] == np.float32(BOX["min_" + a])
        assert got[f"crop_box.max_pt.{i}"] == np.float32(BOX["max_" + a])
    for prefix, field in (("crop_box_", "crop_box.transform"), ("transform_", "transform.matrix")):
        m, want = array(got, field, 12), pose_matrix(POSES[prefix])
        np.testing.assert_allclose(m, want.astype(np.float32), rtol=0, atol=2e-7, err_msg=prefix)
        assert (m[3::4] == want[3::4].astype(np.float32)).all(), prefix
    assert got["frame_id"] == "body"  # transform_target_frame with the transform on
    assert got["publish_cloud"] == 0


def test_empty_launch_gives_the_defaults(harness, tmp_path):
    got = settings(harness, tmp_path, {})
    lib = d2pc.lib()
    assert [got["config." + k] for k in ("fx", "fy", "cx", "cy", "baseline")] == [714.24, 713.5, 376, 240, 0.09]
    cfg = d2pc.default_config()
    assert [got["config." + k] for k in ("fx", "fy", "cx", "cy", "baseline")] == [cfg.fx, cfg.fy, cfg.cx, cfg.cy,
                                                                                  cfg.baseline]
    vox = d2pc.VoxelGrid()
    lib.d2pc_voxel_grid_default(C.byref(vox))
    assert got["voxel_on"] == 0 and got["voxel.leaf_x"] == 0
    for k in ("min_points_per_voxel", "limit_field", "limit_min", "limit_max"):
        assert got["voxel." + k] == getattr(vox, k), k
    assert got["ror_radius"] == 0 and got["ror_min_neighbors"] == 1
    assert got["crop_box.enabled"] == 0 and got["transform.enabled"] == 0
    assert (array(got, "crop_box.min_pt", 3) == -1).all() and (array(got, "crop_box.max_pt", 3) == 1).all()
    identity = np.eye(3, 4).ravel()
    assert (array(got, "crop_box.transform", 12) == identity).all()
    assert (array(got, "transform.matrix", 12) == identity).all()
    for prefix, cls, fn in (("scan", d2pc.LaserScanParams, "d2pc_laser_scan_params_default"),
                            ("map", d2pc.OccupancyParams, "d2pc_occupancy_params_default"),
                            ("projected_map", d2pc.ProjectedMapParams, "d2pc_projected_map_params_default")):
        want = cls()
        getattr(lib, fn)(C.byref(want))
        fields = [f for f, _ in cls._fields_ if f != "struct_size"]
        for f in fields:
            if f == "enabled":
                assert got[f"{prefix}.enabled"] == 0
            elif f == "keep_cloud":
                assert got[f"{prefix}.keep_cloud"] == 1
            else:
                assert got[f"{prefix}.{f}"] == getattr(want, f), (prefix, f)
    assert got["frame_id"] == "/camera_optical_frame" and got["publish_cloud"] == 1


@pytest.mark.parametrize("params,publish", [
    ({"scan_keep_cloud": "0"}, 1), ({"map_keep_cloud": "0"}, 1),  # keep_cloud of a stage that is off
    ({"scan_enable": "1", "scan_keep_cloud": "0"}, 0), ({"map_enable": "1", "map_keep_cloud": "0"}, 0),
    ({"scan_enable": "1", "map_enable": "1"}, 1), ({"transform_target_frame": "body"}, 1)])
def test_publish_cloud_and_frame_id(harness, tmp_path, params, publish):
    got = settings(harness, tmp_path, params)
    assert got["publish_cloud"] == publish
    assert got["frame_id"] == "/camera_optical_frame"  # the transform is off in every case


def test_both_bindings_read_the_params_through_the_shared_reader():
    nodes = os.path.join(ROOT, "include", "d2pc_b200", "nodes.hpp")
    shim = os.path.join(ROOT, "ros1_shim", "disparity_to_point_cloud_node.cpp")
    for path in (nodes, shim):
        assert "d2pc_b200::read_cloud_settings(" in open(path).read(), path
    # each param name is written once: in the reader
    sources = glob.glob(os.path.join(ROOT, "include", "d2pc_b200", "*.hpp")) + \
        glob.glob(os.path.join(ROOT, "ros1_shim", "*.cpp"))
    text = "".join(open(p).read() for p in sources)
    for name in list(PARAMS) + ["voxel_leaf_size", "transform_target_frame"]:
        assert text.count(f'"{name}"') == 1, name
