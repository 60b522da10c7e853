// cloud_stage.cuh -- what the filter stages on clouds already on the device (crop_box.cu, voxel.cu,
// radius_outlier.cu) share: a stage's input and destination, the per-frame bounds pass, and the order-preserving
// compaction.  A batch holds n_frames clouds of at most n_max 16-byte points; position j = f * n_max + i is point i
// of frame f, and a launch takes at most kCloudMaxPoints positions (the caller splits larger batches).
#pragma once
#include <cfloat>
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>
#include <cub/device/device_scan.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

namespace d2pc {

// A stage's input: frame f's points at in + f * in_stride bytes, in_counts[f] of them (values above n_max count as
// n_max; in_counts null: n_max each).  16-byte points, 16-byte aligned.
struct CloudSrc {
  const uint8_t *in = nullptr;
  size_t in_stride = 0;
  const uint32_t *in_counts = nullptr;
  uint32_t n_frames = 0;
  uint32_t n_max = 0;
};

// Where a stage writes a batch's clouds: frame f at points + f * stride, its point count at counts[f].  A compacting
// stage's destination never overlaps its input: kept points are copied after every decision is made.  (The
// transform, a per-point map, may also write exactly over its input.)
struct CloudDst {
  uint8_t *points;
  size_t stride;
  uint32_t *counts;
};

// The sorts and scans index a launch's positions with int, and a scan runs over n_frames * n_max + 1 of them.
constexpr uint64_t kCloudMaxPoints = 0x7ffffffeull;

constexpr int kStageThreads = 256;

inline size_t align_up(size_t v) { return (v + 255) / 256 * 256; }

// bits of the frame number in a sort key
__host__ __device__ __forceinline__ int frame_bits(uint32_t n_frames) {
  int b = 0;
  while ((1ull << b) < n_frames) ++b;
  return b;
}

__device__ __forceinline__ uint32_t frame_count(const CloudSrc &in, uint32_t f) {
  if (!in.in_counts) return in.n_max;
  const uint32_t c = __ldg(in.in_counts + f);
  return c < in.n_max ? c : in.n_max;
}

__device__ __forceinline__ const float4 *frame_points(const CloudSrc &in, uint32_t f) {
  return reinterpret_cast<const float4 *>(in.in + (size_t)f * in.in_stride);
}

// Row a of T * p for a row-major 3x4 [A | t] (t points at the row): ((t[0] * x + t[1] * y) + t[2] * z) + t[3], every
// operation rounded.  Explicit round-to-nearest intrinsics, because nvcc contracts a * b + c to an FMA by default.
// The crop box's local coordinates and the transform stage's output both come from here, so the two cannot drift.
__device__ __forceinline__ float affine_row(const float *t, const float4 &q) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(t[0], q.x), __fmul_rn(t[1], q.y)), __fmul_rn(t[2], q.z)), t[3]);
}

// ---- per-frame bounds: cloud_bounds_kernel (<= kBoundsBlocks blocks over the batch) -> partials, then
// fold_partials at the start of the stage's finish kernel (one block per frame)

struct Partial {
  float mn[3], mx[3], pad[2];
};

__device__ __forceinline__ float warp_min(float v) {
  for (int o = 16; o; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
  for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// min / max of 6 values across the block; the result is valid in thread 0
__device__ __forceinline__ void block_minmax(float (&v)[6]) {
  __shared__ float red[kStageThreads / 32][6];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int a = 0; a < 3; ++a) v[a] = warp_min(v[a]), v[a + 3] = warp_max(v[a + 3]);
  if (lane == 0)
    for (int a = 0; a < 6; ++a) red[warp][a] = v[a];
  __syncthreads();
  if (warp == 0) {
    for (int a = 0; a < 6; ++a) v[a] = lane < kStageThreads / 32 ? red[lane][a] : (a < 3 ? FLT_MAX : -FLT_MAX);
    for (int a = 0; a < 3; ++a) v[a] = warp_min(v[a]), v[a + 3] = warp_max(v[a + 3]);
  }
}

// blocks per frame of the bounds pass: ~8 points per thread, and about kBoundsBlocks blocks over the whole batch
constexpr uint32_t kBoundsBlocks = 1024;
inline uint32_t bounds_blocks(uint32_t n_frames, uint32_t n_max) {
  const uint32_t by_size = (n_max + kStageThreads * 8 - 1) / (kStageThreads * 8);
  const uint32_t by_chip = (kBoundsBlocks + n_frames - 1) / n_frames;
  const uint32_t b = by_size < by_chip ? by_size : by_chip;
  return b ? b : 1;
}

// grid nb * n_frames blocks, frame f's nb blocks consecutive (the frame number on x: a launch takes any number of
// frames): per-block min / max of the points below the frame's count for which pred(point) holds
template <typename Pred>
__global__ void __launch_bounds__(kStageThreads) cloud_bounds_kernel(const CloudSrc in, uint32_t nb, const Pred pred,
                                                                     Partial *__restrict__ partials) {
  const uint32_t f = blockIdx.x / nb, b = blockIdx.x - f * nb, n = frame_count(in, f);
  const float4 *pts = frame_points(in, f);
  float v[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (uint32_t i = b * kStageThreads + threadIdx.x; i < n; i += nb * kStageThreads) {
    const float4 q = __ldg(pts + i);
    if (!pred(q)) continue;
    v[0] = fminf(v[0], q.x), v[1] = fminf(v[1], q.y), v[2] = fminf(v[2], q.z);
    v[3] = fmaxf(v[3], q.x), v[4] = fmaxf(v[4], q.y), v[5] = fmaxf(v[5], q.z);
  }
  block_minmax(v);
  if (threadIdx.x == 0) {
    Partial &o = partials[blockIdx.x];
    for (int a = 0; a < 3; ++a) o.mn[a] = v[a], o.mx[a] = v[a + 3];
  }
}

// frame blockIdx.x's bounds {min xyz, max xyz} from its nb partials, valid in thread 0 (min > max: no point passed)
__device__ __forceinline__ void fold_partials(const Partial *__restrict__ partials, uint32_t nb, float (&v)[6]) {
  const Partial *pp = partials + (size_t)blockIdx.x * nb;
  for (int a = 0; a < 3; ++a) v[a] = FLT_MAX, v[a + 3] = -FLT_MAX;
  for (uint32_t b = threadIdx.x; b < nb; b += kStageThreads)
    for (int a = 0; a < 3; ++a) v[a] = fminf(v[a], pp[b].mn[a]), v[a + 3] = fmaxf(v[a + 3], pp[b].mx[a]);
  block_minmax(v);
}

// ---- the order-preserving compaction: cub::DeviceScan::ExclusiveSum over keep(f, i) of every position, read
// through a transform iterator, gives slot[j] = kept positions before j; cloud_scatter_kernel then copies the kept
// points to their slots and writes the per-frame counts slot[(f + 1) * n_max] - slot[f * n_max].  Keep is a
// device functor of (input, frame f, point index i, position j = f * n_max + i) that returns 1 (kept) or 0, and 0
// at or past the frame's count; a keep that reads only j spares the scan a division per position.  The scatter copies a
// point after keep has decided, so a keep that reads the point shares that load with the copy.

// keep at position j as the scan's uint32 input (0 at j == total: the scan's last slot is the grand total)
template <typename Keep>
struct KeptAt {
  CloudSrc in;
  Keep keep;
  uint32_t total;
  __device__ uint32_t operator()(uint32_t j) const {
    if (j >= total) return 0u;
    const uint32_t f = j / in.n_max;
    return keep(in, f, j - f * in.n_max, j);
  }
};

template <typename Keep>
thrust::transform_iterator<KeptAt<Keep>, thrust::counting_iterator<uint32_t>> kept_positions(const KeptAt<Keep> &k) {
  return thrust::make_transform_iterator(thrust::counting_iterator<uint32_t>(0), k);
}

// grid bpf * n_frames blocks, frame f's bpf blocks consecutive
template <typename Keep>
__global__ void __launch_bounds__(kStageThreads) cloud_scatter_kernel(const CloudSrc in, uint32_t bpf, const Keep keep,
                                                                      const uint32_t *__restrict__ slot,
                                                                      const CloudDst out) {
  const uint32_t f = blockIdx.x / bpf, i = (blockIdx.x - f * bpf) * kStageThreads + threadIdx.x;
  const uint32_t first = f * in.n_max;
  if (i == 0) out.counts[f] = slot[first + in.n_max] - slot[first];
  if (i >= in.n_max || !keep(in, f, i, first + i)) return;
  reinterpret_cast<float4 *>(out.points + (size_t)f * out.stride)[slot[first + i] - slot[first]] =
      __ldg(frame_points(in, f) + i);
}

// the scan's temp storage over n_frames * n_max + 1 positions; the slots take another n_frames * n_max + 1 words
template <typename Keep>
size_t compaction_temp_bytes(uint32_t n_frames, uint32_t n_max) {
  size_t bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, bytes, kept_positions(KeptAt<Keep>{}), (uint32_t *)nullptr,
                                (int)((size_t)n_frames * n_max + 1));
  return bytes;
}

// two launches: the scan (one CUB call) and the scatter
template <typename Keep>
cudaError_t launch_compaction(const CloudSrc &in, const Keep &keep, uint32_t *slot, void *temp, size_t temp_bytes,
                              const CloudDst &out, cudaStream_t stream) {
  const uint32_t total = in.n_frames * in.n_max;
  cudaError_t e = cub::DeviceScan::ExclusiveSum(temp, temp_bytes, kept_positions(KeptAt<Keep>{in, keep, total}),
                                                slot, (int)(total + 1), stream);
  if (e != cudaSuccess) return e;
  const uint32_t bpf = (in.n_max + kStageThreads - 1) / kStageThreads;
  cloud_scatter_kernel<<<bpf * in.n_frames, kStageThreads, 0, stream>>>(in, bpf, keep, slot, out);
  return cudaGetLastError();
}

}  // namespace d2pc
