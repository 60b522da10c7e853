// voxel.cu -- pcl::VoxelGrid<pcl::PointXYZ>::applyFilter (PCL 1.7.2 - 1.12, downsample_all_data = true) on the
// device, batched over frames: the D2PC_FILTER_VOXEL stage behind the CROP kernels.  include/d2pc_b200.h states
// the recipe this file implements; every step there maps onto one stage here:
//
//   1. bounds    voxel_bounds_kernel   per-block min / max of the included points of a frame -> partials
//                                      (positions at or past the frame's input count are excluded like non-finite
//                                      points; no input counts: n each)
//                voxel_finish_kernel   one block per frame: partials -> descriptor (min_b, mul, fallback flag)
//   2. keys      voxel_keys_kernel     (frame << 31 | idx, point index); excluded points sort past every voxel
//   3. sort      cub::DeviceRadixSort::SortPairs on the key bits in use (stable)
//   4. segment   cub::DeviceScan::ExclusiveSum over "voxel head with >= min_points members" -> output slots
//   5. centroid  voxel_centroid_kernel one thread per voxel head folds its members in ascending point index;
//                the same kernel copies the CROP cloud of a fallback frame and writes the per-frame counts
//
// Arithmetic is float32 with explicit round-to-nearest intrinsics (no FMA contraction, no fast-math), as the
// recipe requires; the limit comparison is in double, as PCL compares a float field against double limits.
// No buffer is read before a kernel of the same launch has written it, so the scratch needs no clearing.
#include "voxel.h"

#include <cfloat>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

namespace d2pc {
namespace {

constexpr int kThreads = 256;
constexpr int kFold = 16;  // members loaded per step of the centroid fold
constexpr uint32_t kSentinel = 0x7fffffffu;  // idx of an excluded point: past every voxel (idx <= 2^31 - 2)

struct Desc {
  int32_t min_b[3];
  int32_t fallback;  // 1: the frame's output is its CROP cloud unchanged
  int64_t mul1, mul2;
};

struct Partial {
  float mn[3], mx[3], pad[2];
};

__device__ __forceinline__ bool included(const float4 &q, const VoxelParams &p) {
  if (!(isfinite(q.x) && isfinite(q.y) && isfinite(q.z))) return false;
  if (p.limit_field >= 0) {
    const double v = p.limit_field == 0 ? q.x : (p.limit_field == 1 ? q.y : q.z);
    if (v < p.limit_min || v > p.limit_max) return false;
  }
  return true;
}

// the frame's input count (at most n; no counts: n)
__device__ __forceinline__ uint32_t frame_count(const uint32_t *counts, uint32_t f, uint32_t n) {
  if (!counts) return n;
  const uint32_t c = counts[f];
  return c < n ? c : n;
}

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
  __shared__ float red[kThreads / 32][6];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int a = 0; a < 3; ++a) v[a] = warp_min(v[a]), v[a + 3] = warp_max(v[a + 3]);
  if (lane == 0)
    for (int a = 0; a < 6; ++a) red[warp][a] = v[a];
  __syncthreads();
  if (warp == 0) {
    for (int a = 0; a < 6; ++a) v[a] = lane < kThreads / 32 ? red[lane][a] : (a < 3 ? FLT_MAX : -FLT_MAX);
    for (int a = 0; a < 3; ++a) v[a] = warp_min(v[a]), v[a + 3] = warp_max(v[a + 3]);
  }
}

// grid (blocks_per_frame, n_frames)
__global__ void __launch_bounds__(kThreads) voxel_bounds_kernel(const float4 *__restrict__ crop, uint32_t n,
                                                                const uint32_t *__restrict__ in_counts,
                                                                const VoxelParams p, Partial *__restrict__ partials) {
  const float4 *pts = crop + (size_t)blockIdx.y * n;
  const uint32_t m = frame_count(in_counts, blockIdx.y, n);
  float v[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < m; i += gridDim.x * kThreads) {
    const float4 q = __ldg(pts + i);
    if (!included(q, p)) continue;
    v[0] = fminf(v[0], q.x), v[1] = fminf(v[1], q.y), v[2] = fminf(v[2], q.z);
    v[3] = fmaxf(v[3], q.x), v[4] = fmaxf(v[4], q.y), v[5] = fmaxf(v[5], q.z);
  }
  block_minmax(v);
  if (threadIdx.x == 0) {
    Partial &o = partials[(size_t)blockIdx.y * gridDim.x + blockIdx.x];
    for (int a = 0; a < 3; ++a) o.mn[a] = v[a], o.mx[a] = v[a + 3];
  }
}

// one block per frame: PCL's overflow guard and grid (recipe steps 3-5)
__global__ void __launch_bounds__(kThreads) voxel_finish_kernel(const Partial *__restrict__ partials, uint32_t nb,
                                                                const VoxelParams p, Desc *__restrict__ desc) {
  const Partial *pp = partials + (size_t)blockIdx.x * nb;
  float v[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (uint32_t b = threadIdx.x; b < nb; b += kThreads)
    for (int a = 0; a < 3; ++a) v[a] = fminf(v[a], pp[b].mn[a]), v[a + 3] = fmaxf(v[a + 3], pp[b].mx[a]);
  block_minmax(v);
  if (threadIdx.x != 0) return;
  Desc d = {};
  if (v[0] <= v[3]) {  // at least one included point (otherwise every key is the sentinel: an empty cloud)
    // PCL: dx = (int64)((max_p - min_p) * inv) + 1; dx*dy*dz > INT32_MAX -> output = input.  Evaluated in double,
    // which decides that comparison exactly and also covers spans whose int64 conversion would be undefined.
    double prod = 1.0;
    for (int a = 0; a < 3; ++a) prod *= trunc((double)__fmul_rn(__fsub_rn(v[a + 3], v[a]), p.inv[a])) + 1.0;
    bool fb = !(prod <= 2147483647.0);
    // the grid in PCL's int arithmetic; where that would leave int32 (a bound outside int32, or an index that
    // could reach 2^31 - 1) PCL's result is undefined and the frame takes the same fallback
    double fl[3], span[3], div[3];
    for (int a = 0; a < 3 && !fb; ++a) {
      fl[a] = floorf(__fmul_rn(v[a], p.inv[a]));
      const float hi = floorf(__fmul_rn(v[a + 3], p.inv[a]));
      if (!(fl[a] >= -2147483648.0 && hi < 2147483648.0)) fb = true;
      span[a] = __fsub_rn(hi, (float)fl[a]);  // the largest ijk[a] any point can get
      div[a] = (double)hi - fl[a] + 1.0;
    }
    if (!fb && !(span[0] + span[1] * div[0] + span[2] * div[0] * div[1] < 2147483647.0)) fb = true;
    d.fallback = fb;
    if (!fb) {
      for (int a = 0; a < 3; ++a) d.min_b[a] = (int32_t)fl[a];
      d.mul1 = (int64_t)div[0];
      d.mul2 = (int64_t)div[0] * (int64_t)div[1];
    }
  }
  desc[blockIdx.x] = d;
}

template <typename KeyT>
__global__ void __launch_bounds__(kThreads) voxel_keys_kernel(const float4 *__restrict__ crop, uint32_t n,
                                                              const uint32_t *__restrict__ in_counts,
                                                              uint32_t total, const VoxelParams p,
                                                              const Desc *__restrict__ desc, KeyT *__restrict__ keys,
                                                              uint32_t *__restrict__ vals) {
  const uint32_t j = blockIdx.x * kThreads + threadIdx.x;
  if (j >= total) return;
  const uint32_t f = j / n, i = j - f * n;
  const Desc d = desc[f];
  uint32_t idx = kSentinel;
  const float4 q = i < frame_count(in_counts, f, n) ? __ldg(crop + j) : make_float4(NAN, NAN, NAN, 0.f);
  if (!d.fallback && included(q, p)) {
    const float c[3] = {q.x, q.y, q.z};
    int64_t ijk[3];
    for (int a = 0; a < 3; ++a)
      ijk[a] = (int)__fsub_rn(floorf(__fmul_rn(c[a], p.inv[a])), (float)d.min_b[a]);
    idx = (uint32_t)(ijk[0] + ijk[1] * d.mul1 + ijk[2] * d.mul2);
  }
  keys[j] = ((KeyT)f << 31) | idx;
  vals[j] = i;
}

// position j (sorted order) opens a voxel that is emitted: first of its key, not the sentinel, and at least
// min_points members (the run is sorted, so that is "the key min_points - 1 places on is the same")
template <typename KeyT>
struct HeadFlag {
  const KeyT *keys;
  uint32_t total;
  uint32_t min_points;
  __host__ __device__ uint32_t operator()(uint32_t j) const {
    if (j >= total) return 0;
    const KeyT k = keys[j];
    if ((uint32_t)(k & kSentinel) == kSentinel) return 0;
    if (j > 0 && keys[j - 1] == k) return 0;
    if (min_points > 1) {
      const uint64_t last = (uint64_t)j + min_points - 1;
      if (last >= total || keys[last] != k) return 0;
    }
    return 1;
  }
};

template <typename KeyT>
__global__ void __launch_bounds__(kThreads) voxel_centroid_kernel(const float4 *__restrict__ crop, uint32_t n,
                                                                  const uint32_t *__restrict__ in_counts,
                                                                  uint32_t total, const Desc *__restrict__ desc,
                                                                  const HeadFlag<KeyT> head,
                                                                  const uint32_t *__restrict__ vals,
                                                                  const uint32_t *__restrict__ slot,
                                                                  uint8_t *__restrict__ out, size_t out_stride,
                                                                  uint32_t *__restrict__ counts,
                                                                  uint32_t *__restrict__ fallback) {
  const uint32_t j = blockIdx.x * kThreads + threadIdx.x;
  if (j >= total) return;
  const uint32_t f = j / n, i = j - f * n, first = f * n;
  float4 *dst = reinterpret_cast<float4 *>(out + (size_t)f * out_stride);
  if (desc[f].fallback) {
    const uint32_t m = frame_count(in_counts, f, n);
    if (i < m) dst[i] = __ldg(crop + j);
    if (i == 0) {
      counts[f] = m;
      if (fallback) fallback[f] = 1;
    }
    return;
  }
  if (i == 0) {
    counts[f] = slot[first + n] - slot[first];
    if (fallback) fallback[f] = 0;
  }
  if (!head(j)) return;
  // the fold is serial by contract: ascending point index, which the stable sort left in place.  The adds stay in
  // that order; the loads of kFold members (key, index, point) are issued together ahead of them, so a large voxel
  // costs one memory latency per kFold points instead of two per point.  Loads past the voxel read other points of
  // the same frame and are discarded.
  const float4 *pts = crop + first;
  const KeyT k = head.keys[j];
  const uint32_t end = first + n;
  float sx = 0.f, sy = 0.f, sz = 0.f;
  uint32_t m = j, cnt = 0;
  bool open = true;
  while (open) {
    KeyT kk[kFold];
    float4 q[kFold];
#pragma unroll
    for (int u = 0; u < kFold; ++u) {
      const bool in = m + u < end;
      kk[u] = in ? head.keys[m + u] : ~k;
      q[u] = __ldg(pts + (in ? vals[m + u] : 0u));
    }
#pragma unroll
    for (int u = 0; u < kFold; ++u) {
      open = open && kk[u] == k;
      if (open) sx = __fadd_rn(sx, q[u].x), sy = __fadd_rn(sy, q[u].y), sz = __fadd_rn(sz, q[u].z), ++cnt;
    }
    m += kFold;
  }
  const float c = (float)cnt;
  dst[slot[j] - slot[first]] = make_float4(__fdiv_rn(sx, c), __fdiv_rn(sy, c), __fdiv_rn(sz, c), 1.0f);
}

inline size_t align_up(size_t v) { return (v + 255) / 256 * 256; }

// blocks per frame of the bounds pass: ~8 points per thread, and about kBoundsBlocks blocks over the whole batch
constexpr uint32_t kBoundsBlocks = 1024;
uint32_t bounds_blocks(uint32_t n_frames, uint32_t n) {
  const uint32_t by_size = (n + kThreads * 8 - 1) / (kThreads * 8);
  const uint32_t by_chip = (kBoundsBlocks + n_frames - 1) / n_frames;
  const uint32_t b = by_size < by_chip ? by_size : by_chip;
  return b ? b : 1;
}

int frame_bits(uint32_t n_frames) {
  int b = 0;
  while ((1ull << b) < n_frames) ++b;
  return b;
}

// every buffer of one launch, carved out of the scratch in this order
struct Layout {
  size_t crop, partials, desc, keys_in, keys_out, vals_in, vals_out, slot, temp, temp_bytes, total;
};

template <typename KeyT>
Layout layout(uint32_t n_frames, uint32_t n) {
  const size_t m = (size_t)n_frames * n;
  Layout L;
  size_t o = 0;
  L.crop = o, o += align_up(m * 16);
  L.partials = o, o += align_up((size_t)n_frames * bounds_blocks(n_frames, n) * sizeof(Partial));
  L.desc = o, o += align_up((size_t)n_frames * sizeof(Desc));
  L.keys_in = o, o += align_up(m * sizeof(KeyT));
  L.keys_out = o, o += align_up(m * sizeof(KeyT));
  L.vals_in = o, o += align_up(m * 4);
  L.vals_out = o, o += align_up(m * 4);
  L.slot = o, o += align_up((m + 1) * 4);
  size_t sort_bytes = 0, scan_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (KeyT *)nullptr, (KeyT *)nullptr, (uint32_t *)nullptr,
                                  (uint32_t *)nullptr, (int)m, 0, 31 + frame_bits(n_frames));
  auto flags = thrust::make_transform_iterator(thrust::counting_iterator<uint32_t>(0), HeadFlag<KeyT>{nullptr, 0, 0});
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, flags, (uint32_t *)nullptr, (int)(m + 1));
  L.temp = o;
  L.temp_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
  o += align_up(L.temp_bytes);
  L.total = o;
  return L;
}

template <typename KeyT>
cudaError_t run(const VoxelLaunch &V, cudaStream_t stream, int *launches) {
  const uint32_t total = V.n_frames * V.n;
  const Layout L = layout<KeyT>(V.n_frames, V.n);
  uint8_t *base = static_cast<uint8_t *>(V.scratch);
  const float4 *crop = reinterpret_cast<const float4 *>(base + L.crop);
  Partial *partials = reinterpret_cast<Partial *>(base + L.partials);
  Desc *desc = reinterpret_cast<Desc *>(base + L.desc);
  KeyT *keys_in = reinterpret_cast<KeyT *>(base + L.keys_in), *keys_out = reinterpret_cast<KeyT *>(base + L.keys_out);
  uint32_t *vals_in = reinterpret_cast<uint32_t *>(base + L.vals_in);
  uint32_t *vals_out = reinterpret_cast<uint32_t *>(base + L.vals_out);
  uint32_t *slot = reinterpret_cast<uint32_t *>(base + L.slot);
  void *temp = base + L.temp;

  const uint32_t nb = bounds_blocks(V.n_frames, V.n);
  voxel_bounds_kernel<<<dim3(nb, V.n_frames), kThreads, 0, stream>>>(crop, V.n, V.in_counts, V.p, partials);
  voxel_finish_kernel<<<V.n_frames, kThreads, 0, stream>>>(partials, nb, V.p, desc);
  const uint32_t grid = (total + kThreads - 1) / kThreads;
  voxel_keys_kernel<KeyT><<<grid, kThreads, 0, stream>>>(crop, V.n, V.in_counts, total, V.p, desc, keys_in, vals_in);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  size_t tb = L.temp_bytes;
  e = cub::DeviceRadixSort::SortPairs(temp, tb, keys_in, keys_out, vals_in, vals_out, (int)total, 0,
                                      31 + frame_bits(V.n_frames), stream);
  if (e != cudaSuccess) return e;
  const HeadFlag<KeyT> head{keys_out, total, V.p.min_points};
  tb = L.temp_bytes;
  e = cub::DeviceScan::ExclusiveSum(temp, tb, thrust::make_transform_iterator(thrust::counting_iterator<uint32_t>(0), head),
                                    slot, (int)(total + 1), stream);
  if (e != cudaSuccess) return e;
  voxel_centroid_kernel<KeyT><<<grid, kThreads, 0, stream>>>(crop, V.n, V.in_counts, total, desc, head, vals_out, slot,
                                                             V.out, V.out_stride, V.counts, V.fallback);
  if (launches) *launches = 6;  // four kernels of this file, the sort and the scan (each CUB call counted once)
  return cudaGetLastError();
}

bool narrow_keys(uint32_t n_frames) { return 31 + frame_bits(n_frames) <= 32; }

}  // namespace

size_t voxel_scratch_bytes(uint32_t n_frames, uint32_t n) {
  return narrow_keys(n_frames) ? layout<uint32_t>(n_frames, n).total : layout<uint64_t>(n_frames, n).total;
}

cudaError_t launch_voxel(const VoxelLaunch &L, cudaStream_t stream, int *launches) {
  if (launches) *launches = 0;
  if (L.n_frames == 0) return cudaSuccess;
  if ((uint64_t)L.n_frames * L.n >= (1ull << 31)) return cudaErrorInvalidValue;  // the caller splits larger batches
  if (L.n == 0) {  // no crop: every frame is the empty cloud
    cudaError_t e = cudaMemsetAsync(L.counts, 0, L.n_frames * sizeof(uint32_t), stream);
    if (e == cudaSuccess && L.fallback) e = cudaMemsetAsync(L.fallback, 0, L.n_frames * sizeof(uint32_t), stream);
    return e;
  }
  return narrow_keys(L.n_frames) ? run<uint32_t>(L, stream, launches) : run<uint64_t>(L, stream, launches);
}

}  // namespace d2pc
