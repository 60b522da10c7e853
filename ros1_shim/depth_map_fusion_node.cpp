// ROS1 shim: the reference's depth_map_fusion_node with the per-pixel merge on the GPU (libd2pc_b200.so).
// Built with catkin where roscpp exists (ros1_shim/package.xml, CMakeLists.txt); in the development image it is
// compiled and linked against the API stand-ins of tests/ros_stubs/ (tests/test_ros1_shim.py).
// Subscriptions, the /fused_depth_map publisher, the offset_x / offset_y parameters follow
// include/disparity_to_point_cloud/depth_map_fusion.hpp:97-124, so launch/depth_map_fusion.launch works unchanged.
// Score frames are preprocessed on the GPU as they arrive (Gaussian / Sobel / threshold / Gaussian chain of
// src/depth_map_fusion.cpp:64-99) and cached as the n x n images the reference caches.  The six debug topics
// (depth_map_fusion.hpp:106-117) are published while they have subscribers, colourised on the GPU
// (d2pc_colorize_depth = colorizeDepth, src/depth_map_fusion.cpp:304-358).
#include <ros/ros.h>
#include <sensor_msgs/Image.h>
#include <sensor_msgs/image_encodings.h>

#include <vector>

#include "d2pc_b200.h"
#include "d2pc_b200/node_params.hpp"

namespace {

class DepthMapFusionGpu {
 public:
  DepthMapFusionGpu() : nh_("~") {
    d1_sub_ = nh_.subscribe("/disparity_1", 1, &DepthMapFusionGpu::DisparityCb1, this);
    d2_sub_ = nh_.subscribe("/disparity_2", 1, &DepthMapFusionGpu::DisparityCb2, this);
    s1_sub_ = nh_.subscribe("/matching_score_1", 1, &DepthMapFusionGpu::MatchingScoreCb1, this);
    s2_sub_ = nh_.subscribe("/matching_score_2", 1, &DepthMapFusionGpu::MatchingScoreCb2, this);
    cropped_depth_1_pub_ = nh_.advertise<sensor_msgs::Image>("/cropped_depth_1", 5);
    cropped_depth_2_pub_ = nh_.advertise<sensor_msgs::Image>("/cropped_depth_2", 5);
    cropped_score_1_pub_ = nh_.advertise<sensor_msgs::Image>("/cropped_score_1", 5);
    cropped_score_2_pub_ = nh_.advertise<sensor_msgs::Image>("/cropped_score_2", 5);
    fused_pub_ = nh_.advertise<sensor_msgs::Image>("/fused_depth_map", 5);
    cropped_score_combined_pub_ = nh_.advertise<sensor_msgs::Image>("/combined_score", 5);
    grad_pub_ = nh_.advertise<sensor_msgs::Image>("/gradient", 5);
    d2pc_config cfg;
    d2pc_config_default(&cfg);
    if (!nh_.getParam("offset_x", cfg.offset_x)) ROS_WARN("Failed to load parameter offset_x");
    if (!nh_.getParam("offset_y", cfg.offset_y)) ROS_WARN("Failed to load parameter offset_y");
    const int rc = d2pc_create(&cfg, 0, &ctx_);
    if (rc != D2PC_OK) {
      ROS_FATAL("d2pc_create: %s", d2pc_strerror(rc));
      ros::shutdown();
    }
  }
  ~DepthMapFusionGpu() { d2pc_destroy(ctx_); }

  // publishWithColor (src/depth_map_fusion.cpp:275-302): colour == false is GRAY_SCALE, true is RAINBOW_WITH_BLACK
  void PublishView(const sensor_msgs::ImageConstPtr &m, const uint8_t *mat, uint32_t w, uint32_t h, uint32_t step,
                   ros::Publisher &pub, bool colour) {
    if (pub.getNumSubscribers() == 0) return;
    sensor_msgs::Image out;
    out.header = m->header;
    out.height = h;
    out.width = w;
    out.is_bigendian = 0;
    const uint8_t *src = mat;
    uint32_t src_step = step, row_bytes = w;
    out.encoding = sensor_msgs::image_encodings::MONO8;
    d2pc_image rgb;
    if (colour) {
      if (d2pc_colorize_depth(ctx_, mat, w, h, step, &rgb) != D2PC_OK) return;
      src = rgb.data, src_step = rgb.step, row_bytes = 3 * w;
      out.encoding = sensor_msgs::image_encodings::RGB8;
    }
    out.step = row_bytes;
    d2pc_b200::dense_rows(src, src_step, row_bytes, h, out.data);
    pub.publish(out);
  }
  // cropToSquare(+-offset) [after rotateMat for map 2] as a dense copy -- debug views only
  void PublishCroppedDepth(const sensor_msgs::ImageConstPtr &m, int which, ros::Publisher &pub) {
    if (pub.getNumSubscribers() == 0) return;
    uint32_t n = 0;
    std::vector<uint8_t> v;
    if (d2pc_b200::cropped_view(ctx_, *m, which, v, n) != D2PC_OK) return;
    PublishView(m, v.data(), n, n, n, pub, true);
  }

  void DisparityCb1(const sensor_msgs::ImageConstPtr &m) {
    d1_ = m;
    PublishCroppedDepth(m, 1, cropped_depth_1_pub_);
  }
  void MatchingScoreCb1(const sensor_msgs::ImageConstPtr &m) {
    Preprocess(m, 1, s1_, n1_);
    if (!s1_.empty()) PublishView(m, s1_.data(), n1_, n1_, n1_, cropped_score_1_pub_, false);
  }
  void MatchingScoreCb2(const sensor_msgs::ImageConstPtr &m) {
    Preprocess(m, 2, s2_, n2_);
    if (!s2_.empty()) PublishView(m, s2_.data(), n2_, n2_, n2_, cropped_score_2_pub_, false);
  }
  void Preprocess(const sensor_msgs::ImageConstPtr &m, int which, std::vector<uint8_t> &slot, uint32_t &n) {
    d2pc_image out;
    if (d2pc_preprocess_score(ctx_, m->data.data(), m->width, m->height, m->step, which, &out) != D2PC_OK) return;
    d2pc_b200::dense_rows(out.data, out.step, out.width, out.height, slot);
    n = out.width;
  }
  void DisparityCb2(const sensor_msgs::ImageConstPtr &m) {
    d2_ = m;
    PublishCroppedDepth(m, 2, cropped_depth_2_pub_);
    if (!d1_ || s1_.empty() || s2_.empty()) return;  // have not received all maps and scores yet
    if (d1_->width != m->width || d1_->height != m->height || d1_->step != m->step) return;
    d2pc_image fused, combined;
    const int rc = d2pc_fuse_preprocessed(ctx_, d1_->data.data(), d2_->data.data(), s1_.data(), s2_.data(), m->width,
                                          m->height, m->step, &fused, &combined);
    if (rc != D2PC_OK) {
      ROS_ERROR("d2pc_fuse_preprocessed: %s", d2pc_strerror(rc));
      return;
    }
    // the reference's combined score aliases its cached score 1 (src/depth_map_fusion.cpp:113)
    d2pc_b200::dense_rows(combined.data, combined.step, combined.width, combined.height, s1_);
    sensor_msgs::Image out;
    out.header = m->header;
    out.height = fused.height;
    out.width = fused.width;
    out.encoding = sensor_msgs::image_encodings::MONO8;
    out.is_bigendian = 0;
    out.step = fused.width;
    d2pc_b200::dense_rows(fused.data, fused.step, fused.width, fused.height, out.data);
    PublishView(m, s1_.data(), n1_, n1_, n1_, cropped_score_combined_pub_, false);   // :126-127
    PublishView(m, out.data.data(), out.width, out.height, out.step, grad_pub_, true);  // :132
    fused_pub_.publish(out);
  }

 private:
  ros::NodeHandle nh_;
  ros::Subscriber d1_sub_, d2_sub_, s1_sub_, s2_sub_;
  ros::Publisher fused_pub_, cropped_depth_1_pub_, cropped_depth_2_pub_, cropped_score_1_pub_, cropped_score_2_pub_,
      cropped_score_combined_pub_, grad_pub_;
  sensor_msgs::ImageConstPtr d1_, d2_;
  std::vector<uint8_t> s1_, s2_;  // n x n, dense
  uint32_t n1_ = 0, n2_ = 0;
  d2pc_ctx *ctx_ = nullptr;
};

}  // namespace

int main(int argc, char **argv) {
  ros::init(argc, argv, "depth_map_fusion");
  DepthMapFusionGpu node;
  ros::spin();
  return 0;
}
