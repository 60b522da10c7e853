// laser_scan.h -- host-side launcher interface of laser_scan.cu: the scan pointcloud_to_laserscan would publish for each
// cloud of a batch (the last step of a plan with the scan on, and d2pc_laser_scan_device; the recipe is in
// include/d2pc_b200.h).  Input and batch limit are cloud_stage.cuh's.
#pragma once
#include "cloud_stage.cuh"

namespace d2pc {

// The recipe's settings, decided once per submission (the message's float fields widened where the recipe compares
// against them).
struct LaserScanParams {
  double min_height, max_height;  // the params
  double range_min, range_max;    // the params (double)
  double angle_min, angle_max;    // (double)angle_min_f, (double)angle_max_f
  double angle_increment;         // (double)angle_increment_f
  uint32_t n;                     // ranges per frame
  uint32_t init_bits;             // the initial value of every range, as float bits (>= 0)
};

// Bins shared by a block in shared memory up to this many ranges; larger scans bin into global memory directly.
constexpr uint32_t kScanSharedBins = 4096;

// Frame f's n ranges at ranges + f * ranges_stride bytes (4-byte aligned): two launches, the fill with the initial
// value and the binning of every point below the frame's count.  n == 0 launches nothing.
cudaError_t launch_laser_scan(const CloudSrc &in, const LaserScanParams &p, float *ranges, size_t ranges_stride,
                              cudaStream_t stream, int *launches);

}  // namespace d2pc
