// stand-in for <octomap_msgs/Octomap.h>: see ../ros/ros.h
#pragma once
#include "d2pc_b200/ros_lite.hpp"
namespace octomap_msgs {
using Octomap = ros_lite::octomap_msgs::Octomap;
}  // namespace octomap_msgs
