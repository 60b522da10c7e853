// nodes.hpp -- C++ host mirror of the reference's two node classes, on top of the C ABI (d2pc_b200.h).
//
//   d2pc::Disparity2PCloud            include/disparity_to_point_cloud/disparity_to_point_cloud.hpp:60-109
//   depth_map_fusion::DepthMapFusion  include/disparity_to_point_cloud/depth_map_fusion.hpp:63-155
//
// Same class names, callback names, topic names, queue sizes, latch flag, parameter names and defaults as the
// reference; the bodies hand the pixels to libd2pc_b200.so instead of OpenCV / PCL.  Header-only and ROS-free:
// the topic plumbing is the in-process `Bus` below (what roscpp's single-threaded spin does for one process),
// so the classes run in the offline harness and in tests.  ros1_shim/ shows the same classes bound to a real
// roscpp NodeHandle.  The point cloud node's params, their defaults and the messages it fills come from
// node_params.hpp, which both bindings share.
//
// Deliberate differences from the reference, all at the edges of the hot path:
//   * cv_bridge::toCvCopy(msg, "mono8") converts colour encodings; here only mono8 / 8UC1 are accepted and
//     anything else throws std::invalid_argument (the reference would throw cv_bridge::Exception for encodings
//     it can not convert, src/disparity_to_point_cloud.cpp:50).
//   * the nine printf progress lines per frame (cpp:47-91) are dropped; `verbose` prints "Cloud size: N".
//   * the six debug views of the fusion node are computed only while somebody subscribes to them (a roscpp
//     publisher without subscribers does not serialise either).
#pragma once
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
#include "node_params.hpp"
#include "ros_lite.hpp"

namespace d2pc_b200 {

namespace sensor_msgs = ros_lite::sensor_msgs;

// ---- a process-local stand-in for roscore + roscpp's NodeHandle ------------------------------------------
class Bus {
 public:
  using ImageCb = std::function<void(const sensor_msgs::ImageConstPtr &)>;
  using CloudCb = std::function<void(const sensor_msgs::PointCloud2 &)>;
  using ScanCb = std::function<void(const sensor_msgs::LaserScan &)>;
  using OctomapCb = std::function<void(const ros_lite::octomap_msgs::Octomap &)>;
  using GridCb = std::function<void(const ros_lite::nav_msgs::OccupancyGrid &)>;

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
  void subscribe_octomap(const std::string &topic, uint32_t queue_size, OctomapCb cb) {
    octomap_subs_[resolve(topic)].push_back({queue_size, std::move(cb)});
  }
  void subscribe_grid(const std::string &topic, uint32_t queue_size, GridCb cb) {
    grid_subs_[resolve(topic)].push_back({queue_size, std::move(cb)});
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
  void publish(const std::string &resolved_topic, const ros_lite::octomap_msgs::Octomap &msg) {
    auto it = octomap_subs_.find(resolved_topic);
    if (it != octomap_subs_.end())
      for (auto &s : it->second) s.cb(msg);
  }
  void publish(const std::string &resolved_topic, const ros_lite::nav_msgs::OccupancyGrid &msg) {
    auto it = grid_subs_.find(resolved_topic);
    if (it != grid_subs_.end())
      for (auto &s : it->second) s.cb(msg);
  }
  const std::vector<Advertised> &advertised() const { return advertised_; }
  bool has_subscribers(const std::string &resolved_topic) const {  // ros::Publisher::getNumSubscribers() > 0
    auto it = image_subs_.find(resolved_topic);
    auto ot = octomap_subs_.find(resolved_topic);
    auto gt = grid_subs_.find(resolved_topic);
    return (it != image_subs_.end() && !it->second.empty()) || (ot != octomap_subs_.end() && !ot->second.empty()) ||
           (gt != grid_subs_.end() && !gt->second.empty());
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
  std::map<std::string, std::vector<Sub<OctomapCb>>> octomap_subs_;
  std::map<std::string, std::vector<Sub<GridCb>>> grid_subs_;
  std::map<std::string, sensor_msgs::PointCloud2> latched_clouds_;
  std::vector<Advertised> advertised_;
};

inline void check(int status, const char *what, const d2pc_ctx *ctx = nullptr) {
  if (status != D2PC_OK)
    throw std::runtime_error(std::string(what) + ": " + d2pc_strerror(status) +
                             (ctx ? std::string(" [") + d2pc_last_cuda_error(ctx) + "]" : std::string()));
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
  const d2pc_b200::CloudSettings s_;  // the node's params (node_params.hpp)
  std::string p_cloud_topic_;
  double Q_[16];
  d2pc_ctx *ctx_ = nullptr;
  // The published message is a member, not a local as in the reference (cpp:83): the storage of its data vector
  // is page-locked once (d2pc_b200::reserve_output) and the library DMAs every cloud straight into it.
  sensor_msgs::PointCloud2 output_;
  uint8_t *registered_ = nullptr;
  std::string p_scan_topic_;  // "/scan" with the scan on
  sensor_msgs::LaserScan scan_;
  std::string p_map_topic_;  // "/octomap_point_cloud_centers" with the map on
  sensor_msgs::PointCloud2 centres_;
  std::string p_octomap_topic_[2];  // "/octomap_full", "/octomap_binary" with the map on
  ros_lite::octomap_msgs::Octomap octomap_;
  std::string p_grid_topic_;  // "/projected_map" with the map on
  ros_lite::nav_msgs::OccupancyGrid grid_;

 public:
  explicit Disparity2PCloud(d2pc_b200::Bus &nh, int device = 0, bool verbose = false)
      : nh_(nh), s_(d2pc_b200::read_cloud_settings(nh)) {
    // hpp:77-81: subscribe "/disparity" queue 1; advertise "/point_cloud" queue 1 -- the reference passes `this`
    // as the latch flag, so the publisher is latched.
    nh_.subscribe_image("/disparity", 1, [this](const sensor_msgs::ImageConstPtr &m) { DisparityCb(m); });
    p_cloud_topic_ = nh_.advertise("/point_cloud", 1, /*latch=*/true);
    d2pc_config cfg = s_.config;
    cfg.verbose = verbose ? 1 : 0;
    d2pc_b200::check(d2pc_create(&cfg, device, &ctx_), "d2pc_create");
    d2pc_get_q(ctx_, Q_);
    const char *what = "";
    d2pc_b200::check(d2pc_b200::apply_cloud_settings(ctx_, s_, &what), what, ctx_);
    if (s_.scan.enabled) p_scan_topic_ = nh_.advertise("/scan", 1);
    if (s_.map.enabled) {  // octomap_server's topics, latch false; the octomaps and the grid only while subscribed
      p_map_topic_ = nh_.advertise("/octomap_point_cloud_centers", 1);
      p_octomap_topic_[0] = nh_.advertise("/octomap_full", 1);
      p_octomap_topic_[1] = nh_.advertise("/octomap_binary", 1);
      p_grid_topic_ = nh_.advertise("/projected_map", 1);
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
    const size_t bytes = s_.publish_cloud ? d2pc_b200::crop_bytes(msg->width, msg->height, s_.config.border) : 0;
    d2pc_b200::reserve_output(output_, bytes, registered_);
    d2pc_cloud cloud;
    uint8_t dummy[16];
    uint8_t *dst = output_.data.empty() ? dummy : output_.data.data();
    d2pc_b200::check(d2pc_process_mono8_into(ctx_, msg->data.data(), msg->width, msg->height, msg->step, dst,
                                             output_.data.size(), &cloud),
                     "d2pc_process_mono8_into", ctx_);
    d2pc_b200::describe(cloud, output_);  // pcl::toROSMsg(*cloud, output), cpp:84-85 -- the bytes are already there
    output_.header.stamp = msg->header.stamp;  // cpp:87
    output_.header.frame_id = s_.frame_id;     // cpp:89
    if (s_.publish_cloud) nh_.publish(p_cloud_topic_, output_);  // cpp:90
    if (s_.scan.enabled) {
      d2pc_laser_scan s;
      d2pc_b200::check(d2pc_last_scan(ctx_, &s), "d2pc_last_scan", ctx_);
      d2pc_b200::fill_scan(s, output_.header, scan_);
      nh_.publish(p_scan_topic_, scan_);
    }
    if (!s_.map.enabled) return;
    d2pc_b200::check(d2pc_b200::fetch_centres(ctx_, output_.header, centres_), "d2pc_occupancy_centers", ctx_);
    nh_.publish(p_map_topic_, centres_);
    for (int binary = 0; binary < 2; ++binary) {
      if (!nh_.has_subscribers(p_octomap_topic_[binary])) continue;
      d2pc_octomap m;
      d2pc_b200::check(d2pc_occupancy_octomap(ctx_, binary, &m), "d2pc_occupancy_octomap", ctx_);
      d2pc_b200::fill_octomap(m, output_.header, octomap_);
      nh_.publish(p_octomap_topic_[binary], octomap_);
    }
    if (!nh_.has_subscribers(p_grid_topic_)) return;
    // nothing while the map is empty (publishAll's early return), nor when a padded corner has no key (octomap_server
    // logs an error and publishes no valid grid)
    d2pc_grid_map g;
    const int rc = d2pc_occupancy_projected_map(ctx_, &s_.projected_map, &g);
    if (rc != D2PC_ERR_BAD_DIMS) d2pc_b200::check(rc, "d2pc_occupancy_projected_map", ctx_);
    if (rc == D2PC_OK && g.width) {
      d2pc_b200::fill_grid(g, output_.header, grid_);
      nh_.publish(p_grid_topic_, grid_);
    }
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
    d2pc_b200::dense_rows(out.data, out.step, out.width, out.height, slot);
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
      d2pc_b200::dense_rows(mat, step, w, h, out->data);
    } else {
      d2pc_image rgb;
      d2pc_b200::check(d2pc_colorize_depth(ctx_, mat, w, h, step, &rgb), "d2pc_colorize_depth", ctx_);
      out->encoding = "rgb8";
      out->step = 3 * w;
      d2pc_b200::dense_rows(rgb.data, rgb.step, 3 * w, h, out->data);
    }
    nh_.publish(topic, sensor_msgs::ImageConstPtr(out));
  }

  void publish_cropped_depth(const sensor_msgs::ImageConstPtr &msg, int which, const std::string &topic) {
    if (!nh_.has_subscribers(topic)) return;
    uint32_t n = 0;
    std::vector<uint8_t> v;
    d2pc_b200::check(d2pc_b200::cropped_view(ctx_, *msg, which, v, n), "d2pc_fuse_geometry");
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
      d2pc_b200::dense_rows(m.data.data(), m.step, w, h, tmp);
      return tmp.data();
    };
    std::vector<uint8_t> t1, t2;
    d2pc_image fused, combined;
    d2pc_b200::check(d2pc_fuse_preprocessed(ctx_, dense(depth_1_, t1), dense(depth_2_, t2), cropped_score_1_.data(),
                                            cropped_score_2_.data(), w, h, w, &fused, &combined),
                     "d2pc_fuse_preprocessed", ctx_);
    // :113, :118-121: cropped_score_combined_ aliases cropped_score_1_, so after a fusion pass the cached score 1
    // holds min(score1, score2) until the next MatchingScoreCb1 replaces it.
    d2pc_b200::dense_rows(combined.data, combined.step, dims[0], dims[0], cropped_score_1_);
    // :126-127 the combined score, :132 the colourised fused map (d2pc_colorize_depth reuses the context's
    // output buffers, so the fused pixels are copied out first)
    auto out = std::make_shared<sensor_msgs::Image>();  // disparity->toImageMsg(fused_image), :134-135
    out->header = msg->header;
    out->height = fused.height;
    out->width = fused.width;
    out->encoding = "mono8";
    out->is_bigendian = 0;
    out->step = fused.width;
    d2pc_b200::dense_rows(fused.data, fused.step, fused.width, fused.height, out->data);
    publishWithColor(msg, cropped_score_1_.data(), dims[0], dims[0], dims[0], combined_topic_, GRAY_SCALE);
    publishWithColor(msg, out->data.data(), out->width, out->height, out->step, grad_topic_, RAINBOW_WITH_BLACK);
    nh_.publish(fused_topic_, sensor_msgs::ImageConstPtr(out));  // :136
  }
};

}  // namespace depth_map_fusion
