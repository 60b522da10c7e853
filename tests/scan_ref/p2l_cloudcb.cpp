// PointCloudToLaserScanNodelet::cloudCb (pointcloud_to_laserscan, ROS1 1.4.x) restated from memory, line for line,
// over a cloud that is already in the target frame (test infrastructure, not product code).  It uses glibc's double
// hypot and atan2 (the C functions, float coordinates widened; a float overload would be a different reference), the
// message's float fields and the reference's sequential min.  The one change: a bin
// index at or past the number of ranges is skipped (the reference writes out of bounds there).
//
//   uint32_t d2pc_p2l_cloudcb(const float *pts, size_t n_pts, const double prm[8], int use_inf, float *ranges,
//                             uint32_t cap)
// prm = {min_height, max_height, angle_min, angle_max, angle_increment, range_min, range_max, inf_epsilon}; returns
// ranges.size() and writes the first min(size, cap) ranges.
#include <math.h>

#include <cmath>
#include <cstddef>
#include <cstdint>
#include <limits>
#include <vector>

namespace {
struct LaserScan {
  float angle_min, angle_max, angle_increment, time_increment, scan_time, range_min, range_max;
  std::vector<float> ranges;
};
}  // namespace

extern "C" uint32_t d2pc_p2l_cloudcb(const float *pts, size_t n_pts, const double prm[8], int use_inf,
                                     float *ranges_out, uint32_t cap) {
  const double min_height_ = prm[0], max_height_ = prm[1], angle_min_ = prm[2], angle_max_ = prm[3],
               angle_increment_ = prm[4], range_min_ = prm[5], range_max_ = prm[6], inf_epsilon_ = prm[7];
  const bool use_inf_ = use_inf != 0;
  LaserScan output_;
  LaserScan *output = &output_;
  output->angle_min = angle_min_;
  output->angle_max = angle_max_;
  output->angle_increment = angle_increment_;
  output->time_increment = 0.0;
  output->range_min = range_min_;
  output->range_max = range_max_;
  // determine amount of rays to create
  uint32_t ranges_size = std::ceil((output->angle_max - output->angle_min) / output->angle_increment);
  // determine if laserscan rays with no obstacle data will evaluate to infinity or max_range
  if (use_inf_)
    output->ranges.assign(ranges_size, std::numeric_limits<double>::infinity());
  else
    output->ranges.assign(ranges_size, output->range_max + inf_epsilon_);
  for (size_t i = 0; i < n_pts; ++i) {
    const float *iter_x = pts + 4 * i, *iter_y = pts + 4 * i + 1, *iter_z = pts + 4 * i + 2;
    if (std::isnan(*iter_x) || std::isnan(*iter_y) || std::isnan(*iter_z)) continue;
    if (*iter_z > max_height_ || *iter_z < min_height_) continue;
    double range = ::hypot((double)*iter_x, (double)*iter_y);
    if (range < range_min_) continue;
    if (range > range_max_) continue;
    double angle = ::atan2((double)*iter_y, (double)*iter_x);
    if (angle < output->angle_min || angle > output->angle_max) continue;
    // overwrite range at laserscan ray if new range is smaller
    int index = (angle - output->angle_min) / output->angle_increment;
    if (index < 0 || static_cast<uint32_t>(index) >= ranges_size) continue;  // the reference writes out of bounds
    if (range < output->ranges[index]) output->ranges[index] = range;
  }
  for (uint32_t k = 0; k < ranges_size && k < cap; ++k) ranges_out[k] = output->ranges[k];
  return ranges_size;
}
