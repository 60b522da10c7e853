// nodes.hpp -- C++ host mirror of the reference's two node classes, on top of the C ABI (d2pc_b200.h).
//
//   d2pc::Disparity2PCloud            include/disparity_to_point_cloud/disparity_to_point_cloud.hpp:60-109
//   depth_map_fusion::DepthMapFusion  include/disparity_to_point_cloud/depth_map_fusion.hpp:63-155
//
// Same class names, callback names, topic names, queue sizes, latch flag, parameter names and defaults as the
// reference; the bodies hand the pixels to libd2pc_b200.so instead of OpenCV / PCL.  Header-only and ROS-free:
// the topic plumbing is the in-process `Bus` below (what roscpp's single-threaded spin does for one process),
// so the classes run in the offline harness and in tests.  ros1_shim/ shows the same classes bound to a real
// roscpp NodeHandle.
//
// Deliberate differences from the reference, all at the edges of the hot path:
//   * cv_bridge::toCvCopy(msg, "mono8") converts colour encodings; here only mono8 / 8UC1 are accepted and
//     anything else throws std::invalid_argument (the reference would throw cv_bridge::Exception for encodings
//     it can not convert, src/disparity_to_point_cloud.cpp:50).
//   * the nine printf progress lines per frame (cpp:47-91) are dropped; `verbose` prints "Cloud size: N".
//   * the six debug views of the fusion node are computed only while somebody subscribes to them (a roscpp
//     publisher without subscribers does not serialise either).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <fstream>
#include <functional>
#include <map>
#include <regex>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "../d2pc_b200.h"
#include "ros_lite.hpp"

namespace d2pc_b200 {

namespace sensor_msgs = ros_lite::sensor_msgs;

// ---- a process-local stand-in for roscore + roscpp's NodeHandle ------------------------------------------
class Bus {
 public:
  using ImageCb = std::function<void(const sensor_msgs::ImageConstPtr &)>;
  using CloudCb = std::function<void(const sensor_msgs::PointCloud2 &)>;
  using ScanCb = std::function<void(const sensor_msgs::LaserScan &)>;

  // <remap from="/disparity" to="/throttled_depth_map"/>
  void remap(const std::string &from, const std::string &to) { remaps_[from] = to; }
  std::string resolve(const std::string &name) const {
    auto it = remaps_.find(name);
    return it == remaps_.end() ? name : it->second;
  }
  void set_param(const std::string &name, double v) { params_[name] = v; }
  void set_param(const std::string &name, const std::string &v) { str_params_[name] = v; }
  template <typename T>
  bool get_param(const std::string &name, T &out) const {
    auto it = params_.find(name);
    if (it == params_.end()) return false;
    out = static_cast<T>(it->second);
    return true;
  }
  bool get_param(const std::string &name, std::string &out) const {
    auto it = str_params_.find(name);
    if (it == str_params_.end()) return false;
    out = it->second;
    return true;
  }
  template <typename T>
  void param(const std::string &name, T &out, T def) const {
    if (!get_param(name, out)) out = def;
  }

  void subscribe_image(const std::string &topic, uint32_t queue_size, ImageCb cb) {
    image_subs_[resolve(topic)].push_back({queue_size, std::move(cb)});
  }
  void subscribe_cloud(const std::string &topic, uint32_t queue_size, CloudCb cb) {
    const std::string t = resolve(topic);
    cloud_subs_[t].push_back({queue_size, cb});
    auto it = latched_clouds_.find(t);  // a latched publisher re-delivers its last message to late subscribers
    if (it != latched_clouds_.end()) cb(it->second);
  }
  void subscribe_scan(const std::string &topic, uint32_t queue_size, ScanCb cb) {
    scan_subs_[resolve(topic)].push_back({queue_size, std::move(cb)});
  }
  struct Advertised {
    std::string topic;
    uint32_t queue_size;
    bool latch;
  };
  std::string advertise(const std::string &topic, uint32_t queue_size, bool latch = false) {
    const std::string t = resolve(topic);
    advertised_.push_back({t, queue_size, latch});
    return t;
  }
  void publish(const std::string &resolved_topic, const sensor_msgs::ImageConstPtr &msg) {
    auto it = image_subs_.find(resolved_topic);
    if (it != image_subs_.end())
      for (auto &s : it->second) s.cb(msg);
  }
  void publish(const std::string &resolved_topic, const sensor_msgs::PointCloud2 &msg) {
    for (const auto &a : advertised_)
      if (a.topic == resolved_topic && a.latch) latched_clouds_[resolved_topic] = msg;
    auto it = cloud_subs_.find(resolved_topic);
    if (it != cloud_subs_.end())
      for (auto &s : it->second) s.cb(msg);
  }
  void publish(const std::string &resolved_topic, const sensor_msgs::LaserScan &msg) {
    auto it = scan_subs_.find(resolved_topic);
    if (it != scan_subs_.end())
      for (auto &s : it->second) s.cb(msg);
  }
  const std::vector<Advertised> &advertised() const { return advertised_; }
  bool has_subscribers(const std::string &resolved_topic) const {  // ros::Publisher::getNumSubscribers() > 0
    auto it = image_subs_.find(resolved_topic);
    return it != image_subs_.end() && !it->second.empty();
  }

  // Reads <remap from= to=/> and <param name= value=/> out of a roslaunch file (launch/*.launch).  A value that
  // std::stod reads as a whole (surrounding blanks aside) is a number; any other value is kept as a string.
  bool load_launch_file(const std::string &path) {
    std::ifstream in(path);
    if (!in) return false;
    std::stringstream ss;
    ss << in.rdbuf();
    std::string xml = std::regex_replace(ss.str(), std::regex("<!--[\\s\\S]*?-->"), "");
    auto attr = [](const std::string &tag, const std::string &name) {
      std::smatch m;
      return std::regex_search(tag, m, std::regex(name + "\\s*=\\s*\"([^\"]*)\"")) ? m[1].str() : std::string();
    };
    const std::regex tag_re("<(remap|param)\\b[^>]*>");
    for (auto it = std::sregex_iterator(xml.begin(), xml.end(), tag_re); it != std::sregex_iterator(); ++it) {
      const std::string tag = it->str();
      if ((*it)[1] == "remap")
        remap(attr(tag, "from"), attr(tag, "to"));
      else
        set_launch_param(attr(tag, "name"), attr(tag, "value"));
    }
    return true;
  }

 private:
  void set_launch_param(const std::string &name, const std::string &value) {
    size_t used = 0;
    double v = 0.0;
    try {
      v = std::stod(value, &used);
    } catch (const std::logic_error &) {  // invalid_argument (no number) or out_of_range
      used = 0;
    }
    if (used && value.find_first_not_of(" \t\r\n", used) == std::string::npos)
      set_param(name, v);
    else
      set_param(name, value);
  }

  template <typename Cb>
  struct Sub {
    uint32_t queue_size;
    Cb cb;
  };
  std::map<std::string, std::string> remaps_;
  std::map<std::string, double> params_;
  std::map<std::string, std::string> str_params_;
  std::map<std::string, std::vector<Sub<ImageCb>>> image_subs_;
  std::map<std::string, std::vector<Sub<CloudCb>>> cloud_subs_;
  std::map<std::string, std::vector<Sub<ScanCb>>> scan_subs_;
  std::map<std::string, sensor_msgs::PointCloud2> latched_clouds_;
  std::vector<Advertised> advertised_;
};

inline void check(int status, const char *what, const d2pc_ctx *ctx = nullptr) {
  if (status != D2PC_OK)
    throw std::runtime_error(std::string(what) + ": " + d2pc_strerror(status) +
                             (ctx ? std::string(" [") + d2pc_last_cuda_error(ctx) + "]" : std::string()));
}

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
inline void pose_param(const Bus &nh, const std::string &prefix, float out[12]) {
  const char *names[6] = {"tx", "ty", "tz", "roll", "pitch", "yaw"};
  double pose[6];
  for (int k = 0; k < 6; ++k) nh.param<double>(prefix + names[k], pose[k], 0.0);
  pose_matrix(pose, out);
}

// cv_bridge::toCvCopy(*msg, "mono8") for the encodings this library accepts.
inline void require_mono8(const sensor_msgs::Image &msg) {
  if (msg.encoding != "mono8" && msg.encoding != "8UC1")
    throw std::invalid_argument("unsupported image encoding '" + msg.encoding + "' (mono8 / 8UC1 only)");
  if (msg.step < msg.width || msg.data.size() < static_cast<size_t>(msg.step) * msg.height)
    throw std::invalid_argument("sensor_msgs/Image: step / data size inconsistent");
}

}  // namespace d2pc_b200

// ==========================================================================================================
namespace d2pc {

namespace sensor_msgs = ros_lite::sensor_msgs;

class Disparity2PCloud {
 private:
  d2pc_b200::Bus &nh_;
  std::string p_cloud_topic_;
  // TODO (kept from the reference): import these with the calibration file or camera info topic
  double fx_ = 714.24;
  double fy_ = 713.5;
  double cx_ = 376;
  double cy_ = 240;
  double base_line_ = 0.09;  // Omni-stereo
  double Q_[16];
  d2pc_ctx *ctx_ = nullptr;
  // The published message is a member, not a local as in the reference (cpp:83): the storage of its data vector
  // is page-locked once (d2pc_host_register) and the library DMAs every cloud straight into it, so the memcpy
  // of pcl::toROSMsg (cpp:84-85) has no counterpart here.
  sensor_msgs::PointCloud2 output_;
  uint8_t *registered_ = nullptr;
  int border_ = 40;  // cpp:70,72
  std::string frame_id_ = "/camera_optical_frame";  // cpp:89; transform_target_frame with the transform on
  std::string p_scan_topic_;  // "/scan" when scan_enable != 0
  bool publish_cloud_ = true;  // false with scan_keep_cloud 0: only /scan is published
  sensor_msgs::LaserScan scan_;

  // make output_.data hold `bytes` bytes in page-locked storage without touching bytes it already has
  void reserve_output(size_t bytes) {
    if (output_.data.capacity() < bytes || output_.data.data() != registered_) {
      if (registered_) d2pc_host_unregister(registered_);
      registered_ = nullptr;
      output_.data.clear();
      output_.data.reserve(bytes + bytes / 4 + 4096);
      output_.data.resize(bytes);
      if (d2pc_host_register(output_.data.data(), output_.data.capacity()) == D2PC_OK) registered_ = output_.data.data();
    } else if (output_.data.size() != bytes) {
      output_.data.resize(bytes);  // capacity suffices: the storage (and its registration) stays
    }
  }

 public:
  explicit Disparity2PCloud(d2pc_b200::Bus &nh, int device = 0, bool verbose = false) : nh_(nh) {
    // hpp:77-81: subscribe "/disparity" queue 1; advertise "/point_cloud" queue 1 -- the reference passes `this`
    // as the latch flag, so the publisher is latched.
    nh_.subscribe_image("/disparity", 1, [this](const sensor_msgs::ImageConstPtr &m) { DisparityCb(m); });
    p_cloud_topic_ = nh_.advertise("/point_cloud", 1, /*latch=*/true);
    // hpp:84-88
    nh_.param<double>("fx_", fx_, 714.24);
    nh_.param<double>("fy_", fy_, 713.5);
    nh_.param<double>("cx_", cx_, 376);
    nh_.param<double>("cy_", cy_, 240);
    nh_.param<double>("base_line_", base_line_, 0.09);
    // hpp:90-104: Q from stereoRectify on a fixed 752x480 image size (done inside d2pc_create)
    d2pc_config cfg;
    d2pc_config_default(&cfg);
    cfg.fx = fx_, cfg.fy = fy_, cfg.cx = cx_, cfg.cy = cy_, cfg.baseline = base_line_;
    cfg.verbose = verbose ? 1 : 0;
    border_ = cfg.border;
    d2pc_b200::check(d2pc_create(&cfg, device, &ctx_), "d2pc_create");
    d2pc_get_q(ctx_, Q_);
    // optional, not in the reference: pcl::VoxelGrid on the device (D2PC_FILTER_VOXEL), with a z pass-through
    // limit when voxel_z_min < voxel_z_max.  With the defaults the node publishes what the reference does.
    double leaf = 0.0, z_min = 0.0, z_max = 0.0;
    nh_.param<double>("voxel_leaf_size", leaf, 0.0);
    nh_.param<double>("voxel_z_min", z_min, 0.0);
    nh_.param<double>("voxel_z_max", z_max, 0.0);
    if (leaf > 0.0) {
      d2pc_voxel_grid g;
      d2pc_voxel_grid_default(&g);
      g.leaf_x = g.leaf_y = g.leaf_z = static_cast<float>(leaf);
      if (z_min < z_max) g.limit_field = 2, g.limit_min = z_min, g.limit_max = z_max;
      d2pc_b200::check(d2pc_set_voxel_grid(ctx_, &g), "d2pc_set_voxel_grid", ctx_);
      d2pc_b200::check(d2pc_set_filter_mode(ctx_, D2PC_FILTER_VOXEL), "d2pc_set_filter_mode", ctx_);
    }
    // optional, not in the reference: pcl::RadiusOutlierRemoval on the device behind the filter mode, on when
    // radius_outlier_radius > 0
    double ror_radius = 0.0;
    int ror_min = 1;
    nh_.param<double>("radius_outlier_radius", ror_radius, 0.0);
    nh_.param<int>("radius_outlier_min_neighbors", ror_min, 1);
    if (ror_radius != 0.0) {
      if (ror_min < 0) throw std::runtime_error("radius_outlier_min_neighbors must not be negative");
      d2pc_radius_outlier r;
      d2pc_radius_outlier_default(&r);
      r.radius = ror_radius;
      r.min_neighbors = static_cast<uint32_t>(ror_min);
      d2pc_b200::check(d2pc_set_radius_outlier(ctx_, &r), "d2pc_set_radius_outlier", ctx_);
    }
    // optional, not in the reference: pcl::CropBox on the device in front of VOXEL and the outlier stage, on when
    // crop_box_enable != 0.  The box is crop_box_{min,max}_{x,y,z} in a frame given by a translation and
    // roll / pitch / yaw (crop_box_{tx,ty,tz,roll,pitch,yaw}, radians): this node builds R = Rz(yaw) Ry(pitch) Rx(roll)
    // in double and rounds [R | t] to the library's float matrix.  That conversion is the node's own; the box moves
    // no point, so it leaves the frame_id alone.
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
      d2pc_b200::pose_param(nh_, "crop_box_", b.transform);
      d2pc_b200::check(d2pc_set_crop_box(ctx_, &b), "d2pc_set_crop_box", ctx_);
    }
    // optional, not in the reference: pcl_ros::transformPointCloud on the device as the first cloud stage, on when
    // transform_enable != 0.  transform_{tx,ty,tz,roll,pitch,yaw} is the static camera -> target transform (say a
    // camera -> body extrinsic), built like the crop box's pose; the crop box then lies in the target frame, and
    // the published frame_id is transform_target_frame, as pcl_ros::transformPointCloud sets it.
    int xform_on = 0;
    nh_.param<int>("transform_enable", xform_on, 0);
    if (xform_on) {
      d2pc_cloud_transform t;
      d2pc_cloud_transform_default(&t);
      t.enabled = 1;
      d2pc_b200::pose_param(nh_, "transform_", t.matrix);
      d2pc_b200::check(d2pc_set_cloud_transform(ctx_, &t), "d2pc_set_cloud_transform", ctx_);
      nh_.param<std::string>("transform_target_frame", frame_id_, "base_link");
    }
    // optional, not in the reference: pointcloud_to_laserscan on the device, published on /scan with the cloud's
    // header, on when scan_enable != 0.  scan_<param> are the nodelet's ten params (min_height, max_height,
    // angle_min, angle_max, angle_increment, scan_time, range_min, range_max, use_inf, inf_epsilon) with its defaults;
    // scan_keep_cloud 0 leaves the cloud on the device and /point_cloud unpublished.  The scan needs a z-up frame:
    // set the transform params.
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
      nh_.param<int>("scan_use_inf", s.use_inf, s.use_inf);
      nh_.param<double>("scan_inf_epsilon", s.inf_epsilon, s.inf_epsilon);
      nh_.param<int>("scan_keep_cloud", s.keep_cloud, 1);
      d2pc_b200::check(d2pc_set_laser_scan(ctx_, &s), "d2pc_set_laser_scan", ctx_);
      publish_cloud_ = s.keep_cloud != 0;
      p_scan_topic_ = nh_.advertise("/scan", 1);
    }
  }
  ~Disparity2PCloud() {
    d2pc_destroy(ctx_);  // waits for the device: nothing writes into output_ any more
    if (registered_) d2pc_host_unregister(registered_);
  }
  Disparity2PCloud(const Disparity2PCloud &) = delete;
  Disparity2PCloud &operator=(const Disparity2PCloud &) = delete;

  const double *Q() const { return Q_; }
  d2pc_ctx *context() { return ctx_; }

  // src/disparity_to_point_cloud.cpp:46-92
  void DisparityCb(const sensor_msgs::ImageConstPtr &msg) {
    d2pc_b200::require_mono8(*msg);
    const long cw = static_cast<long>(msg->width) - 2L * border_, ch = static_cast<long>(msg->height) - 2L * border_;
    reserve_output(publish_cloud_ && cw > 0 && ch > 0 ? static_cast<size_t>(cw) * static_cast<size_t>(ch) * 16 : 0);
    d2pc_cloud cloud;
    uint8_t dummy[16];
    uint8_t *dst = output_.data.empty() ? dummy : output_.data.data();
    d2pc_b200::check(d2pc_process_mono8_into(ctx_, msg->data.data(), msg->width, msg->height, msg->step, dst,
                                             output_.data.size(), &cloud),
                     "d2pc_process_mono8_into", ctx_);
    sensor_msgs::PointCloud2 &output = output_;  // pcl::toROSMsg(*cloud, output), cpp:84-85 -- the bytes are already there
    output.height = cloud.height;
    output.width = cloud.width;
    output.fields.clear();
    for (uint32_t i = 0; i < cloud.n_fields; ++i) {
      sensor_msgs::PointField f;
      f.name = cloud.fields[i].name;
      f.offset = cloud.fields[i].offset;
      f.datatype = cloud.fields[i].datatype;
      f.count = cloud.fields[i].count;
      output.fields.push_back(f);
    }
    output.is_bigendian = cloud.is_bigendian;
    output.point_step = cloud.point_step;
    output.row_step = cloud.row_step;
    output.is_dense = cloud.is_dense;
    // CROP_FINITE / VOXEL / the radius outlier stage keep fewer points than the crop holds: shrink the view, never
    // the storage
    output.data.resize(static_cast<size_t>(cloud.row_step) * cloud.height);
    output.header.stamp = msg->header.stamp;             // cpp:87
    output.header.frame_id = frame_id_;                  // cpp:89
    if (publish_cloud_) nh_.publish(p_cloud_topic_, output);  // cpp:90
    if (p_scan_topic_.empty()) return;
    d2pc_laser_scan s;
    d2pc_b200::check(d2pc_last_scan(ctx_, &s), "d2pc_last_scan", ctx_);
    scan_.header = output.header;
    scan_.angle_min = s.angle_min, scan_.angle_max = s.angle_max, scan_.angle_increment = s.angle_increment;
    scan_.time_increment = s.time_increment, scan_.scan_time = s.scan_time;
    scan_.range_min = s.range_min, scan_.range_max = s.range_max;
    scan_.ranges.assign(s.ranges, s.ranges + s.n_ranges);
    nh_.publish(p_scan_topic_, scan_);
  }
};

}  // namespace d2pc

// ==========================================================================================================
namespace depth_map_fusion {

namespace sensor_msgs = ros_lite::sensor_msgs;

class DepthMapFusion {
 private:
  d2pc_b200::Bus &nh_;
  std::string fused_topic_;
  d2pc_ctx *ctx_ = nullptr;
  // the reference caches cropped cv::Mat views (depth_map_fusion.hpp:79-85).  For the depth maps the crop and the
  // rotation are index arithmetic inside the fusion kernel, so the full frames are cached; the scores are cached
  // as the n x n preprocessed images, exactly what cropped_score_{1,2}_ (== cropped_score_{1,2}_grad_) hold.
  sensor_msgs::Image depth_1_, depth_2_;
  std::vector<uint8_t> cropped_score_1_, cropped_score_2_;
  uint32_t score_n_1_ = 0, score_n_2_ = 0;
  bool have_d1_ = false, have_d2_ = false, have_s1_ = false, have_s2_ = false;

  // src/depth_map_fusion.cpp:64-80 / :82-99 on the GPU (d2pc_preprocess_score)
  void preprocess(const sensor_msgs::ImageConstPtr &msg, int which, std::vector<uint8_t> &slot, uint32_t &n, bool &have) {
    d2pc_b200::require_mono8(*msg);
    d2pc_image out;
    d2pc_b200::check(d2pc_preprocess_score(ctx_, msg->data.data(), msg->width, msg->height, msg->step, which, &out),
                     "d2pc_preprocess_score", ctx_);
    n = out.width;
    slot.assign(out.data, out.data + static_cast<size_t>(out.step) * out.height);
    have = true;
  }

  void cache(const sensor_msgs::ImageConstPtr &msg, sensor_msgs::Image &slot, bool &have) {
    d2pc_b200::require_mono8(*msg);
    slot = *msg;
    have = true;
  }

  // ---- the debug views (depth_map_fusion.hpp:106-117, src/depth_map_fusion.cpp:275-302)
  enum { GRAY_SCALE = -1, RAINBOW_WITH_BLACK = -2 };  // depth_map_fusion.hpp:66-67
  std::string cropped_depth_1_topic_, cropped_depth_2_topic_, cropped_score_1_topic_, cropped_score_2_topic_,
      combined_topic_, grad_topic_;

  // publishWithColor (cpp:275-302): GRAY_SCALE publishes the mat as mono8, RAINBOW_WITH_BLACK runs colorizeDepth
  // (cpp:304-358, on the GPU: d2pc_colorize_depth) and labels the result "rgb8" as the reference does.
  void publishWithColor(const sensor_msgs::ImageConstPtr &msg, const uint8_t *mat, uint32_t w, uint32_t h,
                        uint32_t step, const std::string &topic, int colormap) {
    if (!nh_.has_subscribers(topic)) return;
    auto out = std::make_shared<sensor_msgs::Image>();
    out->header = msg->header;
    out->height = h;
    out->width = w;
    out->is_bigendian = 0;
    if (colormap == GRAY_SCALE) {
      out->encoding = "mono8";
      out->step = w;
      out->data.resize(static_cast<size_t>(w) * h);
      for (uint32_t y = 0; y < h; ++y)
        std::copy_n(mat + static_cast<size_t>(y) * step, w, out->data.data() + static_cast<size_t>(y) * w);
    } else {
      d2pc_image rgb;
      d2pc_b200::check(d2pc_colorize_depth(ctx_, mat, w, h, step, &rgb), "d2pc_colorize_depth", ctx_);
      out->encoding = "rgb8";
      out->step = 3 * w;
      out->data.resize(static_cast<size_t>(3) * w * h);
      for (uint32_t y = 0; y < h; ++y)
        std::copy_n(rgb.data + static_cast<size_t>(y) * rgb.step, 3 * w, out->data.data() + static_cast<size_t>(y) * 3 * w);
    }
    nh_.publish(topic, sensor_msgs::ImageConstPtr(out));
  }

  // cropToSquare(image, +-offset) as a dense n x n copy, for the debug views only (the fusion kernel itself never
  // materialises the crop).  which == 2 also applies rotateMat (cpp:268-273): rot(r, c) = src(H-1-c, r).
  std::vector<uint8_t> cropped_view(const sensor_msgs::Image &m, int which, uint32_t &n) {
    int r1[4], r2[4], rc[4], dims[3];
    d2pc_b200::check(d2pc_fuse_geometry(ctx_, m.width, m.height, r1, r2, rc, dims), "d2pc_fuse_geometry");
    n = static_cast<uint32_t>(dims[0]);
    const int *r = which == 1 ? r1 : r2;
    std::vector<uint8_t> v(static_cast<size_t>(n) * n);
    for (uint32_t i = 0; i < n; ++i)
      for (uint32_t j = 0; j < n; ++j)
        v[static_cast<size_t>(i) * n + j] =
            which == 1 ? m.data[static_cast<size_t>(r[1] + i) * m.step + r[0] + j]
                       : m.data[static_cast<size_t>(m.height - 1 - (r[0] + j)) * m.step + r[1] + i];
    return v;
  }
  void publish_cropped_depth(const sensor_msgs::ImageConstPtr &msg, int which, const std::string &topic) {
    if (!nh_.has_subscribers(topic)) return;
    uint32_t n = 0;
    const std::vector<uint8_t> v = cropped_view(*msg, which, n);
    publishWithColor(msg, v.data(), n, n, n, topic, RAINBOW_WITH_BLACK);
  }

 public:
  int offset_x_ = 0;
  int offset_y_ = 0;
  double scaling_factor_ = 1.0;

  explicit DepthMapFusion(d2pc_b200::Bus &nh, int device = 0) : nh_(nh) {
    // depth_map_fusion.hpp:97-104
    nh_.subscribe_image("/disparity_1", 1, [this](const sensor_msgs::ImageConstPtr &m) { DisparityCb1(m); });
    nh_.subscribe_image("/disparity_2", 1, [this](const sensor_msgs::ImageConstPtr &m) { DisparityCb2(m); });
    nh_.subscribe_image("/matching_score_1", 1, [this](const sensor_msgs::ImageConstPtr &m) { MatchingScoreCb1(m); });
    nh_.subscribe_image("/matching_score_2", 1, [this](const sensor_msgs::ImageConstPtr &m) { MatchingScoreCb2(m); });
    // :106-117
    cropped_depth_1_topic_ = nh_.advertise("/cropped_depth_1", 5);
    cropped_depth_2_topic_ = nh_.advertise("/cropped_depth_2", 5);
    cropped_score_1_topic_ = nh_.advertise("/cropped_score_1", 5);
    cropped_score_2_topic_ = nh_.advertise("/cropped_score_2", 5);
    fused_topic_ = nh_.advertise("/fused_depth_map", 5);
    combined_topic_ = nh_.advertise("/combined_score", 5);
    grad_topic_ = nh_.advertise("/gradient", 5);
    // :119-124
    if (!nh_.get_param("offset_x", offset_x_)) std::fprintf(stderr, "[ WARN] Failed to load parameter offset_x\n");
    if (!nh_.get_param("offset_y", offset_y_)) std::fprintf(stderr, "[ WARN] Failed to load parameter offset_y\n");
    d2pc_config cfg;
    d2pc_config_default(&cfg);
    cfg.offset_x = offset_x_;
    cfg.offset_y = offset_y_;
    d2pc_b200::check(d2pc_create(&cfg, device, &ctx_), "d2pc_create");
  }
  ~DepthMapFusion() { d2pc_destroy(ctx_); }
  DepthMapFusion(const DepthMapFusion &) = delete;
  DepthMapFusion &operator=(const DepthMapFusion &) = delete;

  void DisparityCb1(const sensor_msgs::ImageConstPtr &msg) {  // cpp:46-52
    cache(msg, depth_1_, have_d1_);
    publish_cropped_depth(msg, 1, cropped_depth_1_topic_);
  }
  void DisparityCb2(const sensor_msgs::ImageConstPtr &msg) {  // cpp:54-62
    cache(msg, depth_2_, have_d2_);
    publish_cropped_depth(msg, 2, cropped_depth_2_topic_);
    publishFusedDepthMap(msg);
  }
  void MatchingScoreCb1(const sensor_msgs::ImageConstPtr &msg) {  // cpp:64-80
    preprocess(msg, 1, cropped_score_1_, score_n_1_, have_s1_);
    publishWithColor(msg, cropped_score_1_.data(), score_n_1_, score_n_1_, score_n_1_, cropped_score_1_topic_, GRAY_SCALE);
  }
  void MatchingScoreCb2(const sensor_msgs::ImageConstPtr &msg) {  // cpp:82-99
    preprocess(msg, 2, cropped_score_2_, score_n_2_, have_s2_);
    publishWithColor(msg, cropped_score_2_.data(), score_n_2_, score_n_2_, score_n_2_, cropped_score_2_topic_, GRAY_SCALE);
  }

  // src/depth_map_fusion.cpp:103-136
  void publishFusedDepthMap(const sensor_msgs::ImageConstPtr &msg) {
    if (!have_d1_ || !have_d2_ || !have_s1_ || !have_s2_) return;  // :108-111
    const uint32_t w = depth_2_.width, h = depth_2_.height;
    if (depth_1_.width != w || depth_1_.height != h) throw std::invalid_argument("fusion inputs differ in size");
    int r1[4], r2[4], rc[4], dims[3];
    d2pc_b200::check(d2pc_fuse_geometry(ctx_, w, h, r1, r2, rc, dims), "d2pc_fuse_geometry");
    if (score_n_1_ != static_cast<uint32_t>(dims[0]) || score_n_2_ != static_cast<uint32_t>(dims[0]))
      throw std::invalid_argument("cached scores do not match the depth maps' crop");
    // d2pc_fuse_preprocessed wants one common step for the two depth frames: repack if they differ
    auto dense = [&](const sensor_msgs::Image &m, std::vector<uint8_t> &tmp) -> const uint8_t * {
      if (m.step == w) return m.data.data();
      tmp.resize(static_cast<size_t>(w) * h);
      for (uint32_t y = 0; y < h; ++y) std::copy_n(m.data.data() + static_cast<size_t>(y) * m.step, w, tmp.data() + static_cast<size_t>(y) * w);
      return tmp.data();
    };
    std::vector<uint8_t> t1, t2;
    d2pc_image fused, combined;
    d2pc_b200::check(d2pc_fuse_preprocessed(ctx_, dense(depth_1_, t1), dense(depth_2_, t2), cropped_score_1_.data(),
                                            cropped_score_2_.data(), w, h, w, &fused, &combined),
                     "d2pc_fuse_preprocessed", ctx_);
    // :113, :118-121: cropped_score_combined_ aliases cropped_score_1_, so after a fusion pass the cached score 1
    // holds min(score1, score2) until the next MatchingScoreCb1 replaces it.
    for (int i = 0; i < dims[0]; ++i)
      std::copy_n(combined.data + static_cast<size_t>(i) * combined.step, dims[0],
                  cropped_score_1_.data() + static_cast<size_t>(i) * dims[0]);
    // :126-127 the combined score, :132 the colourised fused map (d2pc_colorize_depth reuses the context's
    // output buffers, so the fused pixels are copied out first)
    auto out = std::make_shared<sensor_msgs::Image>();  // disparity->toImageMsg(fused_image), :134-135
    out->header = msg->header;
    out->height = fused.height;
    out->width = fused.width;
    out->encoding = "mono8";
    out->is_bigendian = 0;
    out->step = fused.width;
    out->data.resize(static_cast<size_t>(fused.width) * fused.height);
    for (uint32_t y = 0; y < fused.height; ++y)
      std::copy_n(fused.data + static_cast<size_t>(y) * fused.step, fused.width, out->data.data() + static_cast<size_t>(y) * fused.width);
    publishWithColor(msg, cropped_score_1_.data(), dims[0], dims[0], dims[0], combined_topic_, GRAY_SCALE);
    publishWithColor(msg, out->data.data(), out->width, out->height, out->step, grad_topic_, RAINBOW_WITH_BLACK);
    nh_.publish(fused_topic_, sensor_msgs::ImageConstPtr(out));  // :136
  }
};

}  // namespace depth_map_fusion
