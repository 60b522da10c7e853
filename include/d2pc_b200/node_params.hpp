// node_params.hpp -- what the two bindings of the nodes share: the ROS-free mirror (nodes.hpp) and the roscpp nodes
// (ros1_shim/).  For the point cloud node: its launch params (the one place each name and default is written), the
// library settings they give, and the messages filled from the library's results; for the fusion node: the debug
// views' crop and the dense row copy.  Header-only and ROS-free: templated on the param source (d2pc_b200::Bus or
// ros::NodeHandle, both of which take nh.param(name, value, default)) and on the message types (ros_lite's or the
// genuine sensor_msgs / octomap_msgs / nav_msgs ones, whose members have the same names).  Nothing here logs or
// throws: each binding keeps its own error policy for the statuses returned.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../d2pc_b200.h"

namespace d2pc_b200 {

// [R | t] of a pose param set (the crop box's and the cloud transform's), row-major 3x4 in float:
// R = Rz(yaw) Ry(pitch) Rx(roll) evaluated in double, pose = {tx, ty, tz, roll, pitch, yaw}.
inline void pose_matrix(const double pose[6], float out[12]) {
  const double cr = std::cos(pose[3]), sr = std::sin(pose[3]), cp = std::cos(pose[4]), sp = std::sin(pose[4]);
  const double cy = std::cos(pose[5]), sy = std::sin(pose[5]);
  const double R[3][3] = {{cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr},
                          {sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr},
                          {-sp, cp * sr, cp * cr}};
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) out[4 * i + j] = static_cast<float>(R[i][j]);
    out[4 * i + 3] = static_cast<float>(pose[i]);
  }
}

// the six pose params <prefix>{tx,ty,tz,roll,pitch,yaw} (default 0) as a float [R | t]
template <class NH>
void pose_param(const NH &nh, const std::string &prefix, float out[12]) {
  const char *names[6] = {"tx", "ty", "tz", "roll", "pitch", "yaw"};
  double pose[6];
  for (int k = 0; k < 6; ++k) nh.param(prefix + names[k], pose[k], 0.0);
  pose_matrix(pose, out);
}

// Everything the point cloud node reads from its params.  The library structs start from their d2pc_*_default
// values; `enabled` in them is what the <stage>_enable param says.
struct CloudSettings {
  d2pc_config config;  // d2pc_config_default with the intrinsics fx_, fy_, cx_, cy_, base_line_
  bool voxel_on;       // voxel_leaf_size > 0
  d2pc_voxel_grid voxel;
  double ror_radius;      // radius_outlier_radius: 0 leaves the stage off
  int ror_min_neighbors;  // radius_outlier_min_neighbors: a negative count is refused
  d2pc_crop_box crop_box;
  d2pc_cloud_transform transform;
  d2pc_laser_scan_params scan;
  d2pc_occupancy_params map;
  d2pc_projected_map_params projected_map;
  std::string frame_id;  // the published header.frame_id
  bool publish_cloud;    // false when a scan or map that is on keeps the cloud on the device
};

template <class NH>
CloudSettings read_cloud_settings(const NH &nh) {
  CloudSettings s;
  auto flag = [&nh](const std::string &name) {
    int v = 0;
    nh.param(name, v, 0);
    return v != 0 ? 1 : 0;
  };
  // hpp:84-88 (the reference's TODO: import these with the calibration file or camera info topic).  Q comes from
  // stereoRectify on a fixed 752x480 image size inside d2pc_create (hpp:90-104).
  d2pc_config_default(&s.config);
  nh.param("fx_", s.config.fx, 714.24);
  nh.param("fy_", s.config.fy, 713.5);
  nh.param("cx_", s.config.cx, 376.0);
  nh.param("cy_", s.config.cy, 240.0);
  nh.param("base_line_", s.config.baseline, 0.09);
  // Everything below is optional and not in the reference; with the defaults the node publishes what the reference
  // does.
  // pcl::VoxelGrid on the device (D2PC_FILTER_VOXEL), on when voxel_leaf_size > 0, with a z pass-through limit when
  // voxel_z_min < voxel_z_max.
  double leaf = 0.0, z_min = 0.0, z_max = 0.0;
  nh.param("voxel_leaf_size", leaf, 0.0);
  nh.param("voxel_z_min", z_min, 0.0);
  nh.param("voxel_z_max", z_max, 0.0);
  d2pc_voxel_grid_default(&s.voxel);
  s.voxel_on = leaf > 0.0;
  s.voxel.leaf_x = s.voxel.leaf_y = s.voxel.leaf_z = static_cast<float>(leaf);
  if (z_min < z_max) s.voxel.limit_field = 2, s.voxel.limit_min = z_min, s.voxel.limit_max = z_max;
  // pcl::RadiusOutlierRemoval on the device behind the filter mode, on when radius_outlier_radius != 0.
  nh.param("radius_outlier_radius", s.ror_radius, 0.0);
  nh.param("radius_outlier_min_neighbors", s.ror_min_neighbors, 1);
  // pcl::CropBox on the device in front of VOXEL and the outlier stage, on when crop_box_enable != 0.  The box is
  // crop_box_{min,max}_{x,y,z} in a frame given by a translation and roll / pitch / yaw (crop_box_{tx,ty,tz,roll,
  // pitch,yaw}, radians): pose_param builds R = Rz(yaw) Ry(pitch) Rx(roll) in double and rounds [R | t] to the
  // library's float matrix.  That conversion is the node's own; the box moves no point, so it leaves the frame_id
  // alone.
  d2pc_crop_box_default(&s.crop_box);
  s.crop_box.enabled = flag("crop_box_enable");
  const char *axes[3] = {"x", "y", "z"};
  for (int a = 0; a < 3; ++a) {
    double lo = -1.0, hi = 1.0;
    nh.param(std::string("crop_box_min_") + axes[a], lo, -1.0);
    nh.param(std::string("crop_box_max_") + axes[a], hi, 1.0);
    s.crop_box.min_pt[a] = static_cast<float>(lo), s.crop_box.max_pt[a] = static_cast<float>(hi);
  }
  pose_param(nh, "crop_box_", s.crop_box.transform);
  // pcl_ros::transformPointCloud on the device as the first cloud stage, on when transform_enable != 0.
  // transform_{tx,ty,tz,roll,pitch,yaw} is the static camera -> target transform (say a camera -> body extrinsic; no
  // tf lookup), built like the crop box's pose; the crop box then lies in the target frame, and the published frame_id
  // is transform_target_frame, as pcl_ros::transformPointCloud sets it.
  d2pc_cloud_transform_default(&s.transform);
  s.transform.enabled = flag("transform_enable");
  pose_param(nh, "transform_", s.transform.matrix);
  std::string target;
  nh.param("transform_target_frame", target, std::string("base_link"));
  s.frame_id = s.transform.enabled ? target : "/camera_optical_frame";  // cpp:89
  // pointcloud_to_laserscan on the device, published on /scan with the cloud's header, on when scan_enable != 0.
  // scan_<param> are the nodelet's ten params with its defaults; scan_keep_cloud 0 leaves the cloud on the device and
  // /point_cloud unpublished.  The scan needs a z-up frame: set the transform params.
  d2pc_laser_scan_params_default(&s.scan);
  s.scan.enabled = flag("scan_enable");
  nh.param("scan_min_height", s.scan.min_height, s.scan.min_height);
  nh.param("scan_max_height", s.scan.max_height, s.scan.max_height);
  nh.param("scan_angle_min", s.scan.angle_min, s.scan.angle_min);
  nh.param("scan_angle_max", s.scan.angle_max, s.scan.angle_max);
  nh.param("scan_angle_increment", s.scan.angle_increment, s.scan.angle_increment);
  nh.param("scan_scan_time", s.scan.scan_time, s.scan.scan_time);
  nh.param("scan_range_min", s.scan.range_min, s.scan.range_min);
  nh.param("scan_range_max", s.scan.range_max, s.scan.range_max);
  nh.param("scan_use_inf", s.scan.use_inf, s.scan.use_inf);
  nh.param("scan_inf_epsilon", s.scan.inf_epsilon, s.scan.inf_epsilon);
  nh.param("scan_keep_cloud", s.scan.keep_cloud, 1);
  // octomap_server's insertScan on the device, on when map_enable != 0: every published cloud goes into one occupancy
  // map, whose occupied voxel centres go out on /octomap_point_cloud_centers with the cloud's header after each frame.
  // map_resolution, map_sensor_model_{hit,miss,min,max}, map_occupancy_thres and map_max_range are octomap_server's
  // resolution, sensor_model/* and occupancy params with its defaults; map_max_bricks sizes the device map;
  // map_keep_cloud 0 leaves the cloud on the device and /point_cloud unpublished.  The sensor origin is the
  // transform's translation: set the transform params.  The map also goes out as octomap_msgs/Octomap on
  // /octomap_full and /octomap_binary, and projected to 2-D as nav_msgs/OccupancyGrid on /projected_map;
  // map_occupancy_min_z, map_occupancy_max_z, map_min_x_size and map_min_y_size are octomap_server's
  // occupancy_min_z, occupancy_max_z, min_x_size and min_y_size with its defaults.
  d2pc_occupancy_params_default(&s.map);
  s.map.enabled = flag("map_enable");
  nh.param("map_resolution", s.map.resolution, s.map.resolution);
  nh.param("map_sensor_model_hit", s.map.prob_hit, s.map.prob_hit);
  nh.param("map_sensor_model_miss", s.map.prob_miss, s.map.prob_miss);
  nh.param("map_sensor_model_min", s.map.clamp_min, s.map.clamp_min);
  nh.param("map_sensor_model_max", s.map.clamp_max, s.map.clamp_max);
  nh.param("map_occupancy_thres", s.map.occupancy_thres, s.map.occupancy_thres);
  nh.param("map_max_range", s.map.max_range, s.map.max_range);
  int bricks = static_cast<int>(s.map.max_bricks);
  nh.param("map_max_bricks", bricks, bricks);
  s.map.max_bricks = bricks > 0 ? static_cast<uint32_t>(bricks) : 0u;  // 0 is refused
  nh.param("map_keep_cloud", s.map.keep_cloud, 1);
  d2pc_projected_map_params_default(&s.projected_map);
  nh.param("map_occupancy_min_z", s.projected_map.occupancy_min_z, s.projected_map.occupancy_min_z);
  nh.param("map_occupancy_max_z", s.projected_map.occupancy_max_z, s.projected_map.occupancy_max_z);
  nh.param("map_min_x_size", s.projected_map.min_x_size, s.projected_map.min_x_size);
  nh.param("map_min_y_size", s.projected_map.min_y_size, s.projected_map.min_y_size);
  s.publish_cloud = (!s.scan.enabled || s.scan.keep_cloud) && (!s.map.enabled || s.map.keep_cloud);
  return s;
}

// The settings to a context made from s.config, stage by stage in the node's order; a stage that is off is left
// alone.  Returns the first failing status, with *what naming the failing setter.
inline int apply_cloud_settings(d2pc_ctx *ctx, const CloudSettings &s, const char **what) {
  int rc = D2PC_OK;
  auto fail = [what](const char *name, int status) {
    *what = name;
    return status;
  };
  if (s.voxel_on) {
    if ((rc = d2pc_set_voxel_grid(ctx, &s.voxel)) != D2PC_OK) return fail("d2pc_set_voxel_grid", rc);
    if ((rc = d2pc_set_filter_mode(ctx, D2PC_FILTER_VOXEL)) != D2PC_OK) return fail("d2pc_set_filter_mode", rc);
  }
  if (s.ror_radius != 0.0) {
    if (s.ror_min_neighbors < 0) return fail("a negative radius_outlier_min_neighbors", D2PC_ERR_INVALID_ARG);
    d2pc_radius_outlier r;
    d2pc_radius_outlier_default(&r);
    r.radius = s.ror_radius;
    r.min_neighbors = static_cast<uint32_t>(s.ror_min_neighbors);
    if ((rc = d2pc_set_radius_outlier(ctx, &r)) != D2PC_OK) return fail("d2pc_set_radius_outlier", rc);
  }
  if (s.crop_box.enabled && (rc = d2pc_set_crop_box(ctx, &s.crop_box)) != D2PC_OK) return fail("d2pc_set_crop_box", rc);
  if (s.transform.enabled && (rc = d2pc_set_cloud_transform(ctx, &s.transform)) != D2PC_OK)
    return fail("d2pc_set_cloud_transform", rc);
  if (s.scan.enabled && (rc = d2pc_set_laser_scan(ctx, &s.scan)) != D2PC_OK) return fail("d2pc_set_laser_scan", rc);
  if (s.map.enabled && (rc = d2pc_set_occupancy(ctx, &s.map)) != D2PC_OK) return fail("d2pc_set_occupancy", rc);
  return D2PC_OK;
}

// Bytes of the cloud of a width x height frame: 16 per pixel of the crop inside the border (cpp:70,72), 0 when the
// crop is empty.
inline size_t crop_bytes(uint32_t width, uint32_t height, int border) {
  const long cw = static_cast<long>(width) - 2L * border, ch = static_cast<long>(height) - 2L * border;
  return cw > 0 && ch > 0 ? static_cast<size_t>(cw) * static_cast<size_t>(ch) * 16 : 0;
}

// Makes m.data hold `bytes` bytes in page-locked storage without touching bytes it already has.  `registered` is the
// storage this registered with d2pc_host_register (nullptr for none); its owner unregisters it after d2pc_destroy.
// The library DMAs every cloud straight into that storage, so pcl::toROSMsg's memcpy (cpp:84-85) has no counterpart.
template <class PointCloud2>
void reserve_output(PointCloud2 &m, size_t bytes, uint8_t *&registered) {
  if (m.data.capacity() < bytes || m.data.data() != registered) {
    if (registered) d2pc_host_unregister(registered);
    registered = nullptr;
    m.data.clear();
    m.data.reserve(bytes + bytes / 4 + 4096);
    m.data.resize(bytes);
    if (d2pc_host_register(m.data.data(), m.data.capacity()) == D2PC_OK) registered = m.data.data();
  } else if (m.data.size() != bytes) {
    m.data.resize(bytes);  // capacity suffices: the storage (and its registration) stays
  }
}

// A PointCloud2's fields from the library's d2pc_cloud; data keeps its storage and shows the cloud's bytes
// (CROP_FINITE, VOXEL and the radius outlier stage keep fewer points than the crop holds: the view shrinks, never the
// storage).
template <class PointCloud2>
void describe(const d2pc_cloud &cloud, PointCloud2 &m) {
  m.height = cloud.height;
  m.width = cloud.width;
  m.fields.resize(cloud.n_fields);
  for (uint32_t i = 0; i < cloud.n_fields; ++i) {
    m.fields[i].name = cloud.fields[i].name;
    m.fields[i].offset = cloud.fields[i].offset;
    m.fields[i].datatype = cloud.fields[i].datatype;
    m.fields[i].count = cloud.fields[i].count;
  }
  m.is_bigendian = cloud.is_bigendian;
  m.point_step = cloud.point_step;
  m.row_step = cloud.row_step;
  m.is_dense = cloud.is_dense;
  m.data.resize(static_cast<size_t>(cloud.row_step) * cloud.height);
}

template <class Header, class LaserScan>
void fill_scan(const d2pc_laser_scan &s, const Header &header, LaserScan &m) {
  m.header = header;
  m.angle_min = s.angle_min, m.angle_max = s.angle_max, m.angle_increment = s.angle_increment;
  m.time_increment = s.time_increment, m.scan_time = s.scan_time;
  m.range_min = s.range_min, m.range_max = s.range_max;
  m.ranges.assign(s.ranges, s.ranges + s.n_ranges);
}

// The map's occupied voxel centres after this frame (octomap_server's octomap_point_cloud_centers) into m, whose data
// grows once when the library says it is too small.
template <class Header, class PointCloud2>
int fetch_centres(d2pc_ctx *ctx, const Header &header, PointCloud2 &m) {
  d2pc_cloud c;
  int rc = d2pc_occupancy_centers(ctx, m.data.data(), m.data.size(), &c);
  if (rc == D2PC_ERR_BUFFER_TOO_SMALL) {
    m.data.resize(static_cast<size_t>(c.width) * 16);
    rc = d2pc_occupancy_centers(ctx, m.data.data(), m.data.size(), &c);
  }
  if (rc != D2PC_OK) return rc;
  describe(c, m);
  m.header = header;
  return D2PC_OK;
}

template <class Header, class Octomap>
void fill_octomap(const d2pc_octomap &o, const Header &header, Octomap &m) {
  m.header = header;
  m.binary = static_cast<uint8_t>(o.binary);
  m.id = "OcTree";
  m.resolution = o.resolution;
  m.data.resize(o.size);
  if (o.size) std::memcpy(m.data.data(), o.data, o.size);
}

template <class Header, class OccupancyGrid>
void fill_grid(const d2pc_grid_map &g, const Header &header, OccupancyGrid &m) {
  m.header = header;
  m.info.resolution = g.resolution;
  m.info.width = g.width, m.info.height = g.height;
  m.info.origin.position.x = g.origin_x, m.info.origin.position.y = g.origin_y;
  m.data.assign(g.data, g.data + static_cast<size_t>(g.width) * g.height);
}

// ---- the fusion node ------------------------------------------------------------------------------------------------

// `rows` rows of `row_bytes` bytes, `step` bytes apart from src, as one dense block in dst
inline void dense_rows(const uint8_t *src, size_t step, size_t row_bytes, size_t rows, std::vector<uint8_t> &dst) {
  dst.resize(row_bytes * rows);
  for (size_t y = 0; y < rows; ++y) std::memcpy(dst.data() + y * row_bytes, src + y * step, row_bytes);
}

// cropToSquare(image, +-offset) of a depth map as a dense n x n copy in v, for the debug views only (the fusion kernel
// itself never materialises the crop).  which == 2 also applies rotateMat (src/depth_map_fusion.cpp:268-273):
// rot(r, c) = src(H-1-c, r).  Returns d2pc_fuse_geometry's status.
template <class Image>
int cropped_view(const d2pc_ctx *ctx, const Image &m, int which, std::vector<uint8_t> &v, uint32_t &n) {
  int r1[4], r2[4], rc[4], dims[3];
  const int status = d2pc_fuse_geometry(ctx, m.width, m.height, r1, r2, rc, dims);
  if (status != D2PC_OK) return status;
  n = static_cast<uint32_t>(dims[0]);
  const int *r = which == 1 ? r1 : r2;
  v.resize(static_cast<size_t>(n) * n);
  for (uint32_t i = 0; i < n; ++i)
    for (uint32_t j = 0; j < n; ++j)
      v[static_cast<size_t>(i) * n + j] =
          which == 1 ? m.data[static_cast<size_t>(r[1] + i) * m.step + r[0] + j]
                     : m.data[static_cast<size_t>(m.height - 1 - (r[0] + j)) * m.step + r[1] + i];
  return D2PC_OK;
}

}  // namespace d2pc_b200
