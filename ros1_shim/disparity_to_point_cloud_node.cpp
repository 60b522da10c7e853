// ROS1 shim: the reference's disparity_to_point_cloud_node with DisparityCb's body replaced by libd2pc_b200.so.
// Built with catkin where roscpp exists (ros1_shim/package.xml, CMakeLists.txt); in the development image it is
// compiled and linked against the API stand-ins of tests/ros_stubs/ (tests/test_ros1_shim.py).
// Topic names, queue sizes and the (accidentally) latched publisher follow
// include/disparity_to_point_cloud/disparity_to_point_cloud.hpp:75-106 of the reference; the params, their defaults
// and the messages filled from the library's results are the node mirror's (include/d2pc_b200/node_params.hpp), so
// launch/d2pcloud.launch works unchanged.  This file keeps the roscpp side: subscriptions, publishers and logging.
#include <nav_msgs/OccupancyGrid.h>
#include <octomap_msgs/Octomap.h>
#include <ros/ros.h>
#include <sensor_msgs/Image.h>
#include <sensor_msgs/LaserScan.h>
#include <sensor_msgs/PointCloud2.h>
#include <sensor_msgs/image_encodings.h>

#include "d2pc_b200.h"
#include "d2pc_b200/node_params.hpp"

namespace {

class Disparity2PCloudGpu {
 public:
  Disparity2PCloudGpu() : nh_("~"), s_(d2pc_b200::read_cloud_settings(nh_)) {
    sub_ = nh_.subscribe("/disparity", 1, &Disparity2PCloudGpu::DisparityCb, this);
    pub_ = nh_.advertise<sensor_msgs::PointCloud2>("/point_cloud", 1, /*latch=*/true);
    int device = 0;
    nh_.param<int>("cuda_device", device, 0);
    int rc = d2pc_create(&s_.config, device, &ctx_);
    if (rc != D2PC_OK) {
      ROS_FATAL("d2pc_create: %s", d2pc_strerror(rc));
      ros::shutdown();
      return;
    }
    const char *what = "";
    if ((rc = d2pc_b200::apply_cloud_settings(ctx_, s_, &what)) != D2PC_OK) {
      ROS_FATAL("%s: %s", what, d2pc_strerror(rc));
      ros::shutdown();
      return;
    }
    if (s_.scan.enabled) scan_pub_ = nh_.advertise<sensor_msgs::LaserScan>("/scan", 1);
    if (s_.map.enabled) {
      map_pub_ = nh_.advertise<sensor_msgs::PointCloud2>("/octomap_point_cloud_centers", 1);
      octomap_pub_[0] = nh_.advertise<octomap_msgs::Octomap>("/octomap_full", 1);
      octomap_pub_[1] = nh_.advertise<octomap_msgs::Octomap>("/octomap_binary", 1);
      grid_pub_ = nh_.advertise<nav_msgs::OccupancyGrid>("/projected_map", 1);
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
    const size_t bytes = s_.publish_cloud ? d2pc_b200::crop_bytes(msg->width, msg->height, s_.config.border) : 0;
    d2pc_b200::reserve_output(out_, bytes, registered_);
    uint8_t dummy[16];
    d2pc_cloud cloud;
    int rc = d2pc_process_mono8_into(ctx_, msg->data.data(), msg->width, msg->height, msg->step,
                                     out_.data.empty() ? dummy : out_.data.data(), out_.data.size(), &cloud);
    if (rc != D2PC_OK) {
      ROS_ERROR("d2pc_process_mono8_into: %s (%s)", d2pc_strerror(rc), d2pc_last_cuda_error(ctx_));
      return;
    }
    d2pc_b200::describe(cloud, out_);
    out_.header.stamp = msg->header.stamp;
    out_.header.frame_id = s_.frame_id;
    if (s_.publish_cloud) pub_.publish(out_);
    d2pc_laser_scan s;
    if (s_.scan.enabled && d2pc_last_scan(ctx_, &s) == D2PC_OK) {
      d2pc_b200::fill_scan(s, out_.header, scan_);
      scan_pub_.publish(scan_);
    }
    if (!s_.map.enabled) return;
    if ((rc = d2pc_b200::fetch_centres(ctx_, out_.header, centres_)) != D2PC_OK) {
      ROS_ERROR("d2pc_occupancy_centers: %s (%s)", d2pc_strerror(rc), d2pc_last_cuda_error(ctx_));
      return;
    }
    map_pub_.publish(centres_);
    for (int binary = 0; binary < 2; ++binary) {
      if (octomap_pub_[binary].getNumSubscribers() == 0) continue;
      d2pc_octomap m;
      if ((rc = d2pc_occupancy_octomap(ctx_, binary, &m)) != D2PC_OK) {
        ROS_ERROR("d2pc_occupancy_octomap: %s (%s)", d2pc_strerror(rc), d2pc_last_cuda_error(ctx_));
        return;
      }
      d2pc_b200::fill_octomap(m, out_.header, octomap_);
      octomap_pub_[binary].publish(octomap_);
    }
    if (grid_pub_.getNumSubscribers() == 0) return;
    // nothing while the map is empty (publishAll's early return); a padded corner without a key skips the frame
    d2pc_grid_map g;
    rc = d2pc_occupancy_projected_map(ctx_, &s_.projected_map, &g);
    if (rc == D2PC_ERR_BAD_DIMS) {
      ROS_ERROR("d2pc_occupancy_projected_map: the padded map leaves the key range");
    } else if (rc != D2PC_OK) {
      ROS_ERROR("d2pc_occupancy_projected_map: %s (%s)", d2pc_strerror(rc), d2pc_last_cuda_error(ctx_));
    } else if (g.width) {
      d2pc_b200::fill_grid(g, out_.header, grid_);
      grid_pub_.publish(grid_);
    }
  }

 private:
  ros::NodeHandle nh_;
  const d2pc_b200::CloudSettings s_;  // the node's params
  ros::Subscriber sub_;
  ros::Publisher pub_, scan_pub_, map_pub_, grid_pub_;  // grid_pub_: /projected_map
  ros::Publisher octomap_pub_[2];                      // /octomap_full, /octomap_binary
  octomap_msgs::Octomap octomap_;
  nav_msgs::OccupancyGrid grid_;
  sensor_msgs::PointCloud2 centres_;  // /octomap_point_cloud_centers
  sensor_msgs::LaserScan scan_;
  d2pc_ctx *ctx_ = nullptr;
  sensor_msgs::PointCloud2 out_;  // persistent so that its data storage can stay page-locked
  uint8_t *registered_ = nullptr;
};

}  // namespace

int main(int argc, char **argv) {
  ros::init(argc, argv, "disparity_to_point_cloud");
  Disparity2PCloudGpu node;
  ros::spin();
  return 0;
}
