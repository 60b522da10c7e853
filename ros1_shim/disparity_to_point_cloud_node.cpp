// ROS1 shim: the reference's disparity_to_point_cloud_node with DisparityCb's body replaced by libd2pc_b200.so.
// Built with catkin where roscpp exists (ros1_shim/package.xml, CMakeLists.txt); in the development image it is
// compiled and linked against the API stand-ins of tests/ros_stubs/ (tests/test_ros1_shim.py).
// Topic names, queue sizes, the (accidentally) latched publisher, parameter names and defaults follow
// include/disparity_to_point_cloud/disparity_to_point_cloud.hpp:75-106 of the reference, so
// launch/d2pcloud.launch works unchanged.
#include <ros/ros.h>
#include <sensor_msgs/Image.h>
#include <sensor_msgs/LaserScan.h>
#include <sensor_msgs/PointCloud2.h>
#include <sensor_msgs/image_encodings.h>

#include <cmath>
#include <cstring>
#include <string>

#include "d2pc_b200.h"

namespace {

// The six pose params <prefix>{tx,ty,tz,roll,pitch,yaw} (default 0) as the library's float [R | t]:
// R = Rz(yaw) Ry(pitch) Rx(roll) in double, rounded with t (the node mirror's pose_param, include/d2pc_b200/nodes.hpp).
void pose_param(ros::NodeHandle &nh, const std::string &prefix, float out[12]) {
  double t[3], rpy[3];
  nh.param<double>(prefix + "tx", t[0], 0.0);
  nh.param<double>(prefix + "ty", t[1], 0.0);
  nh.param<double>(prefix + "tz", t[2], 0.0);
  nh.param<double>(prefix + "roll", rpy[0], 0.0);
  nh.param<double>(prefix + "pitch", rpy[1], 0.0);
  nh.param<double>(prefix + "yaw", rpy[2], 0.0);
  const double cr = std::cos(rpy[0]), sr = std::sin(rpy[0]), cp = std::cos(rpy[1]), sp = std::sin(rpy[1]);
  const double cy = std::cos(rpy[2]), sy = std::sin(rpy[2]);
  const double R[3][3] = {{cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr},
                          {sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr},
                          {-sp, cp * sr, cp * cr}};
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) out[4 * i + j] = static_cast<float>(R[i][j]);
    out[4 * i + 3] = static_cast<float>(t[i]);
  }
}

class Disparity2PCloudGpu {
 public:
  Disparity2PCloudGpu() : nh_("~") {
    sub_ = nh_.subscribe("/disparity", 1, &Disparity2PCloudGpu::DisparityCb, this);
    pub_ = nh_.advertise<sensor_msgs::PointCloud2>("/point_cloud", 1, /*latch=*/true);
    d2pc_config cfg;
    d2pc_config_default(&cfg);
    nh_.param<double>("fx_", cfg.fx, 714.24);
    nh_.param<double>("fy_", cfg.fy, 713.5);
    nh_.param<double>("cx_", cfg.cx, 376);
    nh_.param<double>("cy_", cfg.cy, 240);
    nh_.param<double>("base_line_", cfg.baseline, 0.09);
    int device = 0;
    nh_.param<int>("cuda_device", device, 0);
    border_ = cfg.border;
    const int rc = d2pc_create(&cfg, device, &ctx_);
    if (rc != D2PC_OK) {
      ROS_FATAL("d2pc_create: %s", d2pc_strerror(rc));
      ros::shutdown();
      return;
    }
    // optional, not in the reference: pcl::VoxelGrid on the device, with a z pass-through limit when
    // voxel_z_min < voxel_z_max; with the defaults the node publishes what the reference does
    double leaf = 0.0, z_min = 0.0, z_max = 0.0;
    nh_.param<double>("voxel_leaf_size", leaf, 0.0);
    nh_.param<double>("voxel_z_min", z_min, 0.0);
    nh_.param<double>("voxel_z_max", z_max, 0.0);
    if (leaf > 0.0) {
      d2pc_voxel_grid g;
      d2pc_voxel_grid_default(&g);
      g.leaf_x = g.leaf_y = g.leaf_z = static_cast<float>(leaf);
      if (z_min < z_max) g.limit_field = 2, g.limit_min = z_min, g.limit_max = z_max;
      if (d2pc_set_voxel_grid(ctx_, &g) != D2PC_OK || d2pc_set_filter_mode(ctx_, D2PC_FILTER_VOXEL) != D2PC_OK) {
        ROS_FATAL("voxel_leaf_size %g: not a valid voxel grid", leaf);
        ros::shutdown();
      }
    }
    // optional, not in the reference: pcl::RadiusOutlierRemoval on the device behind the filter mode, on when
    // radius_outlier_radius > 0
    double ror_radius = 0.0;
    int ror_min = 1;
    nh_.param<double>("radius_outlier_radius", ror_radius, 0.0);
    nh_.param<int>("radius_outlier_min_neighbors", ror_min, 1);
    if (ror_radius != 0.0) {
      d2pc_radius_outlier r;
      d2pc_radius_outlier_default(&r);
      r.radius = ror_radius;
      r.min_neighbors = static_cast<uint32_t>(ror_min);
      if (ror_min < 0 || d2pc_set_radius_outlier(ctx_, &r) != D2PC_OK) {
        ROS_FATAL("radius_outlier_radius %g / radius_outlier_min_neighbors %d: not a valid setting", ror_radius,
                  ror_min);
        ros::shutdown();
      }
    }
    // optional, not in the reference: pcl::CropBox on the device in front of VOXEL and the outlier stage, on when
    // crop_box_enable != 0; its pose is crop_box_{tx,ty,tz,roll,pitch,yaw} (pose_param).  The box moves no point.
    int box_on = 0;
    nh_.param<int>("crop_box_enable", box_on, 0);
    if (box_on) {
      d2pc_crop_box b;
      d2pc_crop_box_default(&b);
      b.enabled = 1;
      const char *axes[3] = {"x", "y", "z"};
      for (int a = 0; a < 3; ++a) {
        double lo = -1.0, hi = 1.0;
        nh_.param<double>(std::string("crop_box_min_") + axes[a], lo, -1.0);
        nh_.param<double>(std::string("crop_box_max_") + axes[a], hi, 1.0);
        b.min_pt[a] = static_cast<float>(lo), b.max_pt[a] = static_cast<float>(hi);
      }
      pose_param(nh_, "crop_box_", b.transform);
      if (d2pc_set_crop_box(ctx_, &b) != D2PC_OK) {
        ROS_FATAL("crop_box_*: not a valid crop box (min above max, or a non-finite bound or pose)");
        ros::shutdown();
      }
    }
    // optional, not in the reference: pcl_ros::transformPointCloud on the device as the first cloud stage, on when
    // transform_enable != 0.  transform_{tx,ty,tz,roll,pitch,yaw} is a static camera -> target transform (such as a
    // camera -> body extrinsic; no tf lookup); the crop box then lies in the target frame and the published frame_id
    // is transform_target_frame, as pcl_ros::transformPointCloud sets it.
    int xform_on = 0;
    nh_.param<int>("transform_enable", xform_on, 0);
    if (xform_on) {
      d2pc_cloud_transform t;
      d2pc_cloud_transform_default(&t);
      t.enabled = 1;
      pose_param(nh_, "transform_", t.matrix);
      nh_.param<std::string>("transform_target_frame", frame_id_, "base_link");
      if (d2pc_set_cloud_transform(ctx_, &t) != D2PC_OK) {
        ROS_FATAL("transform_*: not a valid transform (a non-finite pose)");
        ros::shutdown();
      }
    }
    // optional, not in the reference: pointcloud_to_laserscan on the device, published on /scan with the cloud's
    // header, on when scan_enable != 0.  scan_<param> are the nodelet's ten params with its defaults; scan_keep_cloud
    // 0 leaves the cloud on the device and /point_cloud unpublished.  The scan needs a z-up frame: set transform_*.
    int scan_on = 0;
    nh_.param<int>("scan_enable", scan_on, 0);
    if (scan_on) {
      d2pc_laser_scan_params s;
      d2pc_laser_scan_params_default(&s);
      s.enabled = 1;
      nh_.param<double>("scan_min_height", s.min_height, s.min_height);
      nh_.param<double>("scan_max_height", s.max_height, s.max_height);
      nh_.param<double>("scan_angle_min", s.angle_min, s.angle_min);
      nh_.param<double>("scan_angle_max", s.angle_max, s.angle_max);
      nh_.param<double>("scan_angle_increment", s.angle_increment, s.angle_increment);
      nh_.param<double>("scan_scan_time", s.scan_time, s.scan_time);
      nh_.param<double>("scan_range_min", s.range_min, s.range_min);
      nh_.param<double>("scan_range_max", s.range_max, s.range_max);
      int use_inf = s.use_inf, keep = 1;
      nh_.param<int>("scan_use_inf", use_inf, use_inf);
      nh_.param<double>("scan_inf_epsilon", s.inf_epsilon, s.inf_epsilon);
      nh_.param<int>("scan_keep_cloud", keep, 1);
      s.use_inf = use_inf, s.keep_cloud = keep;
      if (d2pc_set_laser_scan(ctx_, &s) != D2PC_OK) {
        ROS_FATAL("scan_*: not a valid laser scan setting");
        ros::shutdown();
      } else {
        publish_cloud_ = keep != 0;
        scan_pub_ = nh_.advertise<sensor_msgs::LaserScan>("/scan", 1);
        scan_on_ = true;
      }
    }
  }
  ~Disparity2PCloudGpu() {
    d2pc_destroy(ctx_);
    if (registered_) d2pc_host_unregister(registered_);
  }

  void DisparityCb(const sensor_msgs::ImageConstPtr &msg) {
    namespace enc = sensor_msgs::image_encodings;
    if (msg->encoding != enc::MONO8 && msg->encoding != enc::TYPE_8UC1) {
      ROS_ERROR_THROTTLE(1.0, "unsupported encoding '%s' (mono8 only)", msg->encoding.c_str());
      return;
    }
    // the cloud is DMA'd straight into the message's (page-locked) data vector: no counterpart of the
    // pcl::toROSMsg memcpy (reference cpp:84-85)
    const long cw = static_cast<long>(msg->width) - 2L * border_, ch = static_cast<long>(msg->height) - 2L * border_;
    const size_t bytes = publish_cloud_ && cw > 0 && ch > 0 ? static_cast<size_t>(cw) * static_cast<size_t>(ch) * 16 : 0;
    sensor_msgs::PointCloud2 &out = out_;
    if (out.data.capacity() < bytes || out.data.data() != registered_) {
      if (registered_) d2pc_host_unregister(registered_);
      registered_ = nullptr;
      out.data.clear();
      out.data.reserve(bytes + bytes / 4 + 4096);
      out.data.resize(bytes);
      if (d2pc_host_register(out.data.data(), out.data.capacity()) == D2PC_OK) registered_ = out.data.data();
    } else if (out.data.size() != bytes) {
      out.data.resize(bytes);
    }
    uint8_t dummy[16];
    d2pc_cloud cloud;
    const int rc = d2pc_process_mono8_into(ctx_, msg->data.data(), msg->width, msg->height, msg->step,
                                           out.data.empty() ? dummy : out.data.data(), out.data.size(), &cloud);
    if (rc != D2PC_OK) {
      ROS_ERROR("d2pc_process_mono8_into: %s (%s)", d2pc_strerror(rc), d2pc_last_cuda_error(ctx_));
      return;
    }
    out.height = cloud.height;
    out.width = cloud.width;
    out.fields.resize(cloud.n_fields);
    for (uint32_t i = 0; i < cloud.n_fields; ++i) {
      out.fields[i].name = cloud.fields[i].name;
      out.fields[i].offset = cloud.fields[i].offset;
      out.fields[i].datatype = cloud.fields[i].datatype;
      out.fields[i].count = cloud.fields[i].count;
    }
    out.is_bigendian = cloud.is_bigendian;
    out.point_step = cloud.point_step;
    out.row_step = cloud.row_step;
    out.is_dense = cloud.is_dense;
    out.data.resize(static_cast<size_t>(cloud.row_step) * cloud.height);
    out.header.stamp = msg->header.stamp;
    out.header.frame_id = frame_id_;
    if (publish_cloud_) pub_.publish(out);
    if (!scan_on_) return;
    d2pc_laser_scan s;
    if (d2pc_last_scan(ctx_, &s) != D2PC_OK) return;
    scan_.header = out.header;
    scan_.angle_min = s.angle_min, scan_.angle_max = s.angle_max, scan_.angle_increment = s.angle_increment;
    scan_.time_increment = s.time_increment, scan_.scan_time = s.scan_time;
    scan_.range_min = s.range_min, scan_.range_max = s.range_max;
    scan_.ranges.assign(s.ranges, s.ranges + s.n_ranges);
    scan_pub_.publish(scan_);
  }

 private:
  ros::NodeHandle nh_;
  ros::Subscriber sub_;
  ros::Publisher pub_, scan_pub_;
  bool scan_on_ = false, publish_cloud_ = true;  // scan_enable, scan_keep_cloud
  sensor_msgs::LaserScan scan_;
  d2pc_ctx *ctx_ = nullptr;
  sensor_msgs::PointCloud2 out_;   // persistent so that its data storage can stay page-locked
  uint8_t *registered_ = nullptr;
  int border_ = 40;
  std::string frame_id_ = "/camera_optical_frame";  // transform_target_frame with the transform on
};

}  // namespace

int main(int argc, char **argv) {
  ros::init(argc, argv, "disparity_to_point_cloud");
  Disparity2PCloudGpu node;
  ros::spin();
  return 0;
}
