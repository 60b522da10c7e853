// voxel.cu -- pcl::VoxelGrid<pcl::PointXYZ>::applyFilter (PCL 1.7.2 - 1.12, downsample_all_data = true) on the
// device, batched over frames: the D2PC_FILTER_VOXEL stage behind the CROP kernels or the crop box.
// include/d2pc_b200.h states the recipe this file implements; every step there maps onto one stage here:
//
//   1. bounds    cloud_bounds_kernel   per-block min / max of the included points of a frame -> partials
//                                      (positions at or past the frame's input count are excluded like non-finite
//                                      points)
//                voxel_finish_kernel   one block per frame: partials -> descriptor (min_b, mul, fallback flag)
//   2. keys      voxel_keys_kernel     (frame << 31 | idx, point index); excluded points sort past every voxel
//   3. sort      cub::DeviceRadixSort::SortPairs on the key bits in use (stable)
//   4. segment   cub::DeviceScan::ExclusiveSum over "voxel head with >= min_points members" -> output slots
//   5. centroid  voxel_centroid_kernel one thread per voxel head folds its members in ascending point index;
//                the same kernel copies the input cloud of a fallback frame and writes the per-frame counts
//
// Arithmetic is float32 with explicit round-to-nearest intrinsics (no FMA contraction, no fast-math), as the
// recipe requires; the limit comparison is in double, as PCL compares a float field against double limits.
// No buffer is read before a kernel of the same launch has written it, so the scratch needs no clearing.
#include "voxel.h"

#include <cub/device/device_radix_sort.cuh>

namespace d2pc {
namespace {

constexpr int kFold = 16;  // members loaded per step of the centroid fold
constexpr uint32_t kSentinel = 0x7fffffffu;  // idx of an excluded point: past every voxel (idx <= 2^31 - 2)

struct Desc {
  int32_t min_b[3];
  int32_t fallback;  // 1: the frame's output is its input cloud unchanged
  int64_t mul1, mul2;
};

__device__ __forceinline__ bool included(const float4 &q, const VoxelParams &p) {
  if (!(isfinite(q.x) && isfinite(q.y) && isfinite(q.z))) return false;
  if (p.limit_field >= 0) {
    const double v = p.limit_field == 0 ? q.x : (p.limit_field == 1 ? q.y : q.z);
    if (v < p.limit_min || v > p.limit_max) return false;
  }
  return true;
}

// the bounds pass's predicate
struct Included {
  VoxelParams p;
  __device__ bool operator()(const float4 &q) const { return included(q, p); }
};

// one block per frame: PCL's overflow guard and grid (recipe steps 3-5)
__global__ void __launch_bounds__(kStageThreads) voxel_finish_kernel(const Partial *__restrict__ partials,
                                                                     uint32_t nb, const VoxelParams p,
                                                                     Desc *__restrict__ desc) {
  float v[6];
  fold_partials(partials, nb, v);
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
__global__ void __launch_bounds__(kStageThreads) voxel_keys_kernel(const CloudSrc in, uint32_t total, const VoxelParams p,
                                                                   const Desc *__restrict__ desc,
                                                                   KeyT *__restrict__ keys,
                                                                   uint32_t *__restrict__ vals) {
  const uint32_t j = blockIdx.x * kStageThreads + threadIdx.x;
  if (j >= total) return;
  const uint32_t f = j / in.n_max, i = j - f * in.n_max;
  const Desc d = desc[f];
  uint32_t idx = kSentinel;
  const float4 q = i < frame_count(in, f) ? __ldg(frame_points(in, f) + i) : make_float4(NAN, NAN, NAN, 0.f);
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
__global__ void __launch_bounds__(kStageThreads) voxel_centroid_kernel(const CloudSrc in, uint32_t total,
                                                                       const Desc *__restrict__ desc,
                                                                       const HeadFlag<KeyT> head,
                                                                       const uint32_t *__restrict__ vals,
                                                                       const uint32_t *__restrict__ slot,
                                                                       const CloudDst out,
                                                                       uint32_t *__restrict__ fallback) {
  const uint32_t j = blockIdx.x * kStageThreads + threadIdx.x;
  if (j >= total) return;
  const uint32_t n = in.n_max, f = j / n, i = j - f * n, first = f * n;
  float4 *dst = reinterpret_cast<float4 *>(out.points + (size_t)f * out.stride);
  if (desc[f].fallback) {
    const uint32_t m = frame_count(in, f);
    if (i < m) dst[i] = __ldg(frame_points(in, f) + i);
    if (i == 0) {
      out.counts[f] = m;
      if (fallback) fallback[f] = 1;
    }
    return;
  }
  if (i == 0) {
    out.counts[f] = slot[first + n] - slot[first];
    if (fallback) fallback[f] = 0;
  }
  if (!head(j)) return;
  // the fold is serial by contract: ascending point index, which the stable sort left in place.  The adds stay in
  // that order; the loads of kFold members (key, index, point) are issued together ahead of them, so a large voxel
  // costs one memory latency per kFold points instead of two per point.  Loads past the voxel read other points of
  // the same frame and are discarded.
  // frame_points(in, f), written from `first`: with the base as f * in_stride nvcc hoists all kFold point loads
  // ahead of the adds (108 registers for 64-bit keys, 2 blocks per SM, a 15-30 % slower stage on a B200); this form
  // keeps the schedule of a dense input (34 registers)
  const float4 *pts =
      reinterpret_cast<const float4 *>(in.in + (size_t)first * 16 + (size_t)f * (in.in_stride - (size_t)n * 16));
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
      const bool own = m + u < end;
      kk[u] = own ? head.keys[m + u] : ~k;
      q[u] = __ldg(pts + (own ? vals[m + u] : 0u));
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

// every buffer of one launch, carved out of the scratch in this order
struct Layout {
  size_t partials, desc, keys_in, keys_out, vals_in, vals_out, slot, temp, temp_bytes, total;
};

template <typename KeyT>
Layout layout(uint32_t n_frames, uint32_t n) {
  const size_t m = (size_t)n_frames * n;
  Layout L;
  size_t o = 0;
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
cudaError_t run(const CloudSrc &in, const CloudDst &out, const VoxelParams &p, uint32_t *fallback, void *scratch,
                cudaStream_t stream, int *launches) {
  const uint32_t total = in.n_frames * in.n_max;
  const Layout L = layout<KeyT>(in.n_frames, in.n_max);
  uint8_t *base = static_cast<uint8_t *>(scratch);
  Partial *partials = reinterpret_cast<Partial *>(base + L.partials);
  Desc *desc = reinterpret_cast<Desc *>(base + L.desc);
  KeyT *keys_in = reinterpret_cast<KeyT *>(base + L.keys_in), *keys_out = reinterpret_cast<KeyT *>(base + L.keys_out);
  uint32_t *vals_in = reinterpret_cast<uint32_t *>(base + L.vals_in);
  uint32_t *vals_out = reinterpret_cast<uint32_t *>(base + L.vals_out);
  uint32_t *slot = reinterpret_cast<uint32_t *>(base + L.slot);
  void *temp = base + L.temp;

  const uint32_t nb = bounds_blocks(in.n_frames, in.n_max);
  cloud_bounds_kernel<<<nb * in.n_frames, kStageThreads, 0, stream>>>(in, nb, Included{p}, partials);
  voxel_finish_kernel<<<in.n_frames, kStageThreads, 0, stream>>>(partials, nb, p, desc);
  const uint32_t grid = (total + kStageThreads - 1) / kStageThreads;
  voxel_keys_kernel<KeyT><<<grid, kStageThreads, 0, stream>>>(in, total, p, desc, keys_in, vals_in);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  size_t tb = L.temp_bytes;
  e = cub::DeviceRadixSort::SortPairs(temp, tb, keys_in, keys_out, vals_in, vals_out, (int)total, 0,
                                      31 + frame_bits(in.n_frames), stream);
  if (e != cudaSuccess) return e;
  const HeadFlag<KeyT> head{keys_out, total, p.min_points};
  tb = L.temp_bytes;
  e = cub::DeviceScan::ExclusiveSum(temp, tb, thrust::make_transform_iterator(thrust::counting_iterator<uint32_t>(0), head),
                                    slot, (int)(total + 1), stream);
  if (e != cudaSuccess) return e;
  voxel_centroid_kernel<KeyT><<<grid, kStageThreads, 0, stream>>>(in, total, desc, head, vals_out, slot, out,
                                                                  fallback);
  if (launches) *launches = 6;  // four kernels of this file, the sort and the scan (each CUB call counted once)
  return cudaGetLastError();
}

bool narrow_keys(uint32_t n_frames) { return 31 + frame_bits(n_frames) <= 32; }

}  // namespace

size_t voxel_scratch_bytes(uint32_t n_frames, uint32_t n_max) {
  return narrow_keys(n_frames) ? layout<uint32_t>(n_frames, n_max).total : layout<uint64_t>(n_frames, n_max).total;
}

cudaError_t launch_voxel(const CloudSrc &in, const CloudDst &out, const VoxelParams &p, uint32_t *fallback,
                         void *scratch, cudaStream_t stream, int *launches) {
  if (launches) *launches = 0;
  if (in.n_frames == 0) return cudaSuccess;
  if ((uint64_t)in.n_frames * in.n_max > kCloudMaxPoints) return cudaErrorInvalidValue;  // the caller splits the batch
  if (in.n_max == 0) {  // no crop: every frame is the empty cloud
    cudaError_t e = cudaMemsetAsync(out.counts, 0, in.n_frames * sizeof(uint32_t), stream);
    if (e == cudaSuccess && fallback) e = cudaMemsetAsync(fallback, 0, in.n_frames * sizeof(uint32_t), stream);
    return e;
  }
  return narrow_keys(in.n_frames) ? run<uint32_t>(in, out, p, fallback, scratch, stream, launches)
                                  : run<uint64_t>(in, out, p, fallback, scratch, stream, launches);
}

}  // namespace d2pc
