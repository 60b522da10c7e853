// stand-in for <nav_msgs/OccupancyGrid.h>: see ../ros/ros.h
#pragma once
#include "d2pc_b200/ros_lite.hpp"
namespace nav_msgs {
using OccupancyGrid = ros_lite::nav_msgs::OccupancyGrid;
}  // namespace nav_msgs
