// stand-in for <sensor_msgs/LaserScan.h>: see ../ros/ros.h
#pragma once
#include "d2pc_b200/ros_lite.hpp"
namespace sensor_msgs {
using LaserScan = ros_lite::sensor_msgs::LaserScan;
}  // namespace sensor_msgs
