// crop_box.cu -- pcl::CropBox<pcl::PointXYZ> (setTransform only, setNegative(false), keep_organized false) on the
// device, batched over frames: the stage in front of VOXEL and the radius outlier stage when a box is enabled, and
// d2pc_crop_box_device.  include/d2pc_b200.h states the recipe.  The stage is a predicate and an order-preserving
// compaction, in two launches:
//
//   1. slots    cub::DeviceScan::ExclusiveSum over "position j is kept", read through a transform iterator that
//               evaluates the predicate on the point (no flag array): slot[j] = kept positions before j
//   2. scatter  crop_box_scatter_kernel  the predicate again; kept points copied unchanged to their slot, and the
//               per-frame counts slot[(f + 1) * n_max] - slot[f * n_max]
//
// Position j = f * n_max + i is point i of frame f; positions at or past the frame's count are not kept.  The local
// coordinates are float32 with explicit round-to-nearest intrinsics, because nvcc contracts a * b + c to an FMA by
// default and the recipe rounds every operation.  No buffer is read before a kernel of the same launch has written
// it, so the scratch needs no clearing.
#include "crop_box.h"

#include <cub/device/device_scan.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

namespace d2pc {
namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ uint32_t frame_count(const uint32_t *counts, uint32_t f, uint32_t n_max) {
  if (!counts) return n_max;
  const uint32_t c = counts[f];
  return c < n_max ? c : n_max;
}

// rows a of l = T * p: ((t[a][0] * x + t[a][1] * y) + t[a][2] * z) + t[a][3], every operation rounded
__device__ __forceinline__ float local(const float *t, const float4 &q) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(t[0], q.x), __fmul_rn(t[1], q.y)), __fmul_rn(t[2], q.z)), t[3]);
}

// recipe rules 1-3: finite, then min <= l <= max on every axis (a NaN l fails)
__device__ __forceinline__ bool inside(const float4 &q, const CropBoxParams &b) {
  if (!(isfinite(q.x) && isfinite(q.y) && isfinite(q.z))) return false;
  bool in = true;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float l = local(b.t + 4 * a, q);
    in = in && b.mn[a] <= l && l <= b.mx[a];
  }
  return in;
}

// "position j is kept" as the scan's uint32 input (0 at j == total: the scan's last slot is the grand total)
struct KeptAt {
  const uint8_t *in;
  size_t in_stride;
  const uint32_t *in_counts;
  uint32_t n_max, total;
  CropBoxParams box;
  __device__ uint32_t operator()(uint32_t j) const {
    if (j >= total) return 0u;
    const uint32_t f = j / n_max, i = j - f * n_max;
    if (i >= frame_count(in_counts, f, n_max)) return 0u;
    return inside(__ldg(reinterpret_cast<const float4 *>(in + (size_t)f * in_stride) + i), box);
  }
};

// grid bpf * n_frames blocks, frame f's bpf blocks consecutive (the frame number on x: no 65535-frame limit)
__global__ void __launch_bounds__(kThreads) crop_box_scatter_kernel(const uint8_t *__restrict__ in, size_t in_stride,
                                                                    const uint32_t *__restrict__ in_counts,
                                                                    uint32_t n_max, uint32_t bpf,
                                                                    const CropBoxParams box,
                                                                    const uint32_t *__restrict__ slot,
                                                                    uint8_t *__restrict__ out, size_t out_stride,
                                                                    uint32_t *__restrict__ counts) {
  const uint32_t f = blockIdx.x / bpf, i = (blockIdx.x - f * bpf) * kThreads + threadIdx.x;
  const uint32_t first = f * n_max;
  if (i == 0) counts[f] = slot[first + n_max] - slot[first];
  if (i >= frame_count(in_counts, f, n_max)) return;
  const float4 q = __ldg(reinterpret_cast<const float4 *>(in + (size_t)f * in_stride) + i);
  if (!inside(q, box)) return;
  reinterpret_cast<float4 *>(out + (size_t)f * out_stride)[slot[first + i] - slot[first]] = q;
}

inline size_t align_up(size_t v) { return (v + 255) / 256 * 256; }

size_t scan_temp_bytes(uint32_t n_frames, uint32_t n_max) {
  const size_t m = (size_t)n_frames * n_max;
  size_t bytes = 0;
  auto kept = thrust::make_transform_iterator(thrust::counting_iterator<uint32_t>(0), KeptAt{});
  cub::DeviceScan::ExclusiveSum(nullptr, bytes, kept, (uint32_t *)nullptr, (int)(m + 1));
  return bytes;
}

}  // namespace

size_t crop_box_scratch_bytes(uint32_t n_frames, uint32_t n_max) {
  return align_up(((size_t)n_frames * n_max + 1) * 4) + align_up(scan_temp_bytes(n_frames, n_max));
}

size_t crop_box_stage_bytes(uint32_t n_frames, uint32_t n) {
  return align_up((size_t)n_frames * n * 16) + align_up((size_t)n_frames * 4) + crop_box_scratch_bytes(n_frames, n);
}

CropBoxStage crop_box_stage(void *buffer, uint32_t n_frames, uint32_t n) {
  uint8_t *b = static_cast<uint8_t *>(buffer);
  const size_t clouds = align_up((size_t)n_frames * n * 16);
  return CropBoxStage{b, reinterpret_cast<uint32_t *>(b + clouds), b + clouds + align_up((size_t)n_frames * 4)};
}

cudaError_t launch_crop_box(const CropBoxLaunch &L, cudaStream_t stream, int *launches) {
  if (launches) *launches = 0;
  if (L.n_frames == 0) return cudaSuccess;
  if ((uint64_t)L.n_frames * L.n_max > kCropBoxMaxPoints) return cudaErrorInvalidValue;  // the caller splits the batch
  if (L.n_max == 0) return cudaMemsetAsync(L.counts, 0, L.n_frames * sizeof(uint32_t), stream);
  const uint32_t total = L.n_frames * L.n_max;
  uint8_t *base = static_cast<uint8_t *>(L.scratch);
  uint32_t *slot = reinterpret_cast<uint32_t *>(base);
  void *temp = base + align_up(((size_t)total + 1) * 4);
  size_t tb = scan_temp_bytes(L.n_frames, L.n_max);
  const KeptAt kept{L.in, L.in_stride, L.in_counts, L.n_max, total, L.box};
  cudaError_t e = cub::DeviceScan::ExclusiveSum(
      temp, tb, thrust::make_transform_iterator(thrust::counting_iterator<uint32_t>(0), kept), slot, (int)(total + 1),
      stream);
  if (e != cudaSuccess) return e;
  const uint32_t bpf = (L.n_max + kThreads - 1) / kThreads;
  crop_box_scatter_kernel<<<bpf * L.n_frames, kThreads, 0, stream>>>(L.in, L.in_stride, L.in_counts, L.n_max, bpf,
                                                                      L.box, slot, L.out, L.out_stride, L.counts);
  if (launches) *launches = 2;  // the scan (one CUB call counted once) and the scatter
  return cudaGetLastError();
}

}  // namespace d2pc
