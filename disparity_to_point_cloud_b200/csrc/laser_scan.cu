// laser_scan.cu -- pointcloud_to_laserscan's binning on the device, batched over frames: the last step of a plan with
// the scan on, and d2pc_laser_scan_device.  include/d2pc_b200.h states the recipe; range and angle are scan_math.h's,
// the source the C reference compiles too.
//
// Two launches.  laser_scan_fill_kernel writes the initial value into every bin of every frame.  laser_scan_bin_kernel
// reads each point below its frame's count with one 16-byte streaming load, applies the recipe's tests and folds
// (float)r into bin k with an atomicMin on the float's bits: every value is >= 0, where unsigned order is float order,
// and the min over a bin's points is the reference's sequential result in any order (the header's argument).  Up to
// kScanSharedBins bins a block folds into its own copy of the frame's bins in shared memory and merges the bins it
// touched with global atomicMin; above that it folds into global memory.  A wall in front of the camera sends the
// lanes of a warp to a few bins; a warp pre-reduction (__match_any_sync + __reduce_min_sync) before the atomics was
// measured slower on such a wall than the plain atomics (DESIGN.md section 2.11), so there is none.  No scratch, no
// ticket.
#include "laser_scan.h"
#include "scan_math.h"

namespace d2pc {
namespace {

constexpr uint32_t kNone = 0xffffffffu;  // "no value": above the bits of every float >= 0, +inf included

__device__ __forceinline__ uint32_t *frame_bins(float *ranges, size_t stride, uint32_t f) {
  return reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(ranges) + (size_t)f * stride);
}

__global__ void __launch_bounds__(kStageThreads) laser_scan_fill_kernel(float *__restrict__ ranges, size_t stride,
                                                                        uint32_t n, uint32_t bpf, uint32_t init) {
  const uint32_t f = blockIdx.x / bpf, k = (blockIdx.x - f * bpf) * kStageThreads + threadIdx.x;
  if (k < n) frame_bins(ranges, stride, f)[k] = init;
}

// The recipe's per-point tests; the bin of an accepted point in *k and its (float)r bits in *v.
__device__ __forceinline__ bool scan_point(const float4 &q, const LaserScanParams &p, uint32_t *k, uint32_t *v) {
  if (isnan(q.x) || isnan(q.y) || isnan(q.z)) return false;
  const double z = (double)q.z;
  if (z > p.max_height || z < p.min_height) return false;
  const double r = d2pc_scan_range(q.x, q.y);
  if (r < p.range_min || r > p.range_max) return false;
  const double a = d2pc_scan_angle((double)q.y, (double)q.x);
  if (a < p.angle_min || a > p.angle_max) return false;
  const int b = (int)__ddiv_rn(__dsub_rn(a, p.angle_min), p.angle_increment);
  if ((uint32_t)b >= p.n) return false;
  *k = (uint32_t)b;
  *v = __float_as_uint(__double2float_rn(r));
  return true;
}

// grid nb * n_frames blocks, frame f's nb blocks consecutive; each block strides over its frame's points
template <bool kShared>
__global__ void __launch_bounds__(kStageThreads) laser_scan_bin_kernel(const CloudSrc in, uint32_t nb,
                                                                       const LaserScanParams p,
                                                                       float *__restrict__ ranges, size_t stride) {
  __shared__ uint32_t sbins[kShared ? kScanSharedBins : 1];
  const uint32_t f = blockIdx.x / nb, b = blockIdx.x - f * nb, n = frame_count(in, f);
  uint32_t *const gbins = frame_bins(ranges, stride, f);
  if (kShared) {
    for (uint32_t k = threadIdx.x; k < p.n; k += kStageThreads) sbins[k] = kNone;
    __syncthreads();
  }
  const float4 *pts = frame_points(in, f);
  for (uint32_t i = b * kStageThreads + threadIdx.x; i < n; i += nb * kStageThreads) {
    uint32_t k, v;
    if (scan_point(__ldcs(pts + i), p, &k, &v)) atomicMin((kShared ? sbins : gbins) + k, v);
  }
  if (kShared) {
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < p.n; k += kStageThreads)
      if (sbins[k] != kNone) atomicMin(gbins + k, sbins[k]);
  }
}

}  // namespace

cudaError_t launch_laser_scan(const CloudSrc &in, const LaserScanParams &p, float *ranges, size_t ranges_stride,
                              cudaStream_t stream, int *launches) {
  if (launches) *launches = 0;
  if (in.n_frames == 0 || p.n == 0) return cudaSuccess;
  if ((uint64_t)in.n_frames * in.n_max > kCloudMaxPoints) return cudaErrorInvalidValue;  // the caller splits the batch
  const uint32_t fill_bpf = (p.n + kStageThreads - 1) / kStageThreads;
  laser_scan_fill_kernel<<<fill_bpf * in.n_frames, kStageThreads, 0, stream>>>(ranges, ranges_stride, p.n, fill_bpf,
                                                                               p.init_bits);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (launches) *launches = 1;
  if (in.n_max == 0) return cudaSuccess;
  // ~16 points per thread: a block's shared bins are cleared and merged once per 4096 points
  const uint32_t nb = bounds_blocks(in.n_frames, (in.n_max + 1) / 2);
  if (p.n <= kScanSharedBins)
    laser_scan_bin_kernel<true><<<nb * in.n_frames, kStageThreads, 0, stream>>>(in, nb, p, ranges, ranges_stride);
  else
    laser_scan_bin_kernel<false><<<nb * in.n_frames, kStageThreads, 0, stream>>>(in, nb, p, ranges, ranges_stride);
  e = cudaGetLastError();
  if (launches && e == cudaSuccess) *launches = 2;
  return e;
}

}  // namespace d2pc
