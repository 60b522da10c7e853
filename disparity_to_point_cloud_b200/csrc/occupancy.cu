// occupancy.cu -- octomap_server's insertScan on the device: the occupancy map behind every host entry with the map
// on, and d2pc_occupancy_insert_device.  include/d2pc_b200.h states the recipe; keys, norms and rays are map_math.h's,
// the source the C reference compiles too.
//
// A frame is three launches on one stream.
//   mark   one thread per point walks computeRayKeys from the origin and marks each free cell with atomicMax(mark,
//          epoch * 4 + 2), then the endpoint's cell with epoch * 4 + 3, so a hit beats a miss in any order and a mark of
//          an older epoch never needs clearing.  The mark is read first and the atomic skipped when it already holds
//          at least that value: every ray crosses the origin's cells.  A thread looks its brick up once per brick it
//          enters, creating it on first use with one atomicCAS on the slot's key (the slot owns the brick's storage,
//          so the loser of a race reads the winner's key and goes on).  The first thread to touch a slot in this epoch
//          appends it to the touched list.  A brick beyond max_bricks, or a table with no free slot on the probe path,
//          sets the overflow flag.
//   apply  one block per touched slot: each voxel marked in this epoch gets its one hit or miss, with octomap's early
//          abort and clamp; nothing at all when the overflow flag is set, so a dropped frame leaves the known map as
//          it was.
//   finish one thread: counts the frame as applied or dropped and clears the flag and the touched count.
#include <cub/device/device_radix_sort.cuh>

#include "map_math.h"
#include "occupancy.h"

namespace d2pc {
namespace {

constexpr uint32_t kNoSlot = 0xffffffffu;
constexpr int kApplyThreads = 256;  // two voxels per thread, one mask word per warp and half-brick

__device__ __forceinline__ unsigned long long brick_key(const uint16_t k[3]) {
  return (unsigned long long)(k[0] >> 3) | ((unsigned long long)(k[1] >> 3) << 16) |
         ((unsigned long long)(k[2] >> 3) << 32);
}
__device__ __forceinline__ uint32_t voxel_in_brick(const uint16_t k[3]) {
  return (k[0] & 7u) | ((k[1] & 7u) << 3) | ((k[2] & 7u) << 6);
}
__device__ __forceinline__ uint32_t slot_hash(unsigned long long bk, uint32_t cap) {
  return (uint32_t)((bk * 0x9E3779B97F4A7C15ull) >> 32) & (cap - 1);
}

// The slot of brick bk, created on first use; kNoSlot (and the overflow flag) when the map cannot take it.
__device__ uint32_t find_slot(const MapTable &t, unsigned long long bk) {
  uint32_t h = slot_hash(bk, t.cap);
  for (uint32_t i = 0; i < t.cap; ++i, h = (h + 1) & (t.cap - 1)) {
    const unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(t.keys + h);
    if (cur == bk) return h;
    if (cur != kMapEmpty) continue;
    if (*reinterpret_cast<volatile uint32_t *>(t.ctr) >= t.max_bricks) {
      // the map is full, but the creator of the last brick may have put it in this very slot after the read above:
      // it wrote the key before it counted the brick (the fence below), so the key is visible here now
      __threadfence();
      const unsigned long long again = *reinterpret_cast<volatile unsigned long long *>(t.keys + h);
      if (again == bk) return h;
      if (again == kMapEmpty) break;
      continue;
    }
    const unsigned long long prev = atomicCAS(t.keys + h, kMapEmpty, bk);
    if (prev == kMapEmpty) {
      // created: the storage is the slot's own; a brick past max_bricks still drops the frame
      __threadfence();
      if (atomicAdd(t.ctr, 1u) >= t.max_bricks) atomicExch(t.ctr + 1, 1u);
      return h;
    }
    if (prev == bk) return h;
  }
  atomicExch(t.ctr + 1, 1u);
  return kNoSlot;
}

// Marks voxel k with v, looking its brick up when the ray enters a new one (*bk / *slot cache the last brick, a
// brick the map could not take included: false then, and nothing is marked -- the frame is dropped anyway).
__device__ __forceinline__ bool mark_voxel(const MapTable &t, const uint16_t k[3], uint32_t v, uint32_t epoch,
                                           unsigned long long *bk, uint32_t *slot) {
  const unsigned long long b = brick_key(k);
  if (b != *bk) {
    *bk = b;
    *slot = find_slot(t, b);
    if (*slot != kNoSlot && t.slot_epoch[*slot] != epoch && atomicExch(t.slot_epoch + *slot, epoch) != epoch)
      t.touched[atomicAdd(t.ctr + 2, 1u)] = *slot;
  }
  if (*slot == kNoSlot) return false;
  uint32_t *m = t.marks + (size_t)*slot * 512 + voxel_in_brick(k);
  if (*m < v) atomicMax(m, v);
  return true;
}

__global__ void __launch_bounds__(kStageThreads) map_mark_kernel(const CloudSrc in, const MapTable t,
                                                                 const MapUpdate u) {
  const uint32_t i = blockIdx.x * kStageThreads + threadIdx.x;
  if (i >= frame_count(in, 0)) return;
  const float4 q = __ldcs(frame_points(in, 0) + i);
  if (!isfinite(q.x) || !isfinite(q.y) || !isfinite(q.z)) return;
  const float p[3] = {q.x, q.y, q.z};
  float e[3];
  int hit;
  d2pc_map_ray_end(u.origin, p, u.max_range, e, &hit);
  const uint32_t miss_mark = u.epoch * 4u + 2u, hit_mark = u.epoch * 4u + 3u;
  unsigned long long bk = kMapEmpty;
  uint32_t slot = kNoSlot;
  d2pc_map_ray r;
  if (d2pc_map_ray_begin(&r, u.origin, e, u.res, u.rf)) {
    bool ok = mark_voxel(t, r.key, miss_mark, u.epoch, &bk, &slot);
    while (ok && d2pc_map_ray_next(&r)) ok = mark_voxel(t, r.key, miss_mark, u.epoch, &bk, &slot);
  }
  uint16_t k[3];
  if (hit && d2pc_map_key3(u.rf, p[0], p[1], p[2], k)) mark_voxel(t, k, hit_mark, u.epoch, &bk, &slot);
}

// grid-stride over the touched slots, one block per slot
__global__ void __launch_bounds__(kApplyThreads) map_apply_kernel(const MapTable t, const MapUpdate u) {
  if (*reinterpret_cast<volatile uint32_t *>(t.ctr + 1)) return;  // overflow: the frame is dropped
  const uint32_t n = t.ctr[2], lane = threadIdx.x & 31;
  for (uint32_t b = blockIdx.x; b < n; b += gridDim.x) {
    const size_t slot = t.touched[b];
    for (int half = 0; half < 2; ++half) {
      const uint32_t i = threadIdx.x + half * kApplyThreads;
      const uint32_t m = t.marks[slot * 512 + i];
      uint32_t *const kw = t.known + slot * 16 + (i >> 5);
      const uint32_t word = *kw;
      const bool known = (word >> lane) & 1u;
      bool created = false;
      if ((m >> 2) == u.epoch) {
        const float up = (m & 1u) ? u.hit : u.miss;
        float *const pv = t.log_odds + slot * 512 + i;
        const float v = known ? *pv : 0.0f;
        // OccupancyOcTreeBase::updateNode's early abort, then addValue and the clamp
        if (!(known && ((up >= 0.0f && v >= u.clamp_max) || (up <= 0.0f && v <= u.clamp_min)))) {
          float w = __fadd_rn(v, up);
          if (w < u.clamp_min) w = u.clamp_min;
          if (w > u.clamp_max) w = u.clamp_max;
          *pv = w;
          created = !known;
        }
      }
      const uint32_t fresh = __ballot_sync(0xffffffffu, created);
      if (lane == 0 && fresh) *kw = word | fresh;
    }
  }
}

__global__ void map_finish_kernel(const MapTable t) {
  ++t.frames[t.ctr[1] ? 1 : 0];
  t.ctr[1] = 0;
  t.ctr[2] = 0;
}

// ---- export

__device__ __forceinline__ bool exported(const MapTable &t, size_t slot, uint32_t i, bool occupied_only,
                                         float thres) {
  if (!((t.known[slot * 16 + (i >> 5)] >> (i & 31)) & 1u)) return false;
  return !occupied_only || t.log_odds[slot * 512 + i] >= thres;
}

__global__ void __launch_bounds__(kApplyThreads) map_count_kernel(const MapTable t, bool occupied_only, float thres,
                                                                  uint32_t *n) {
  for (uint32_t slot = blockIdx.x; slot < t.cap; slot += gridDim.x) {
    if (t.keys[slot] == kMapEmpty) continue;  // uniform across the block
    const int c = __syncthreads_count(exported(t, slot, threadIdx.x, occupied_only, thres)) +
                  __syncthreads_count(exported(t, slot, threadIdx.x + kApplyThreads, occupied_only, thres));
    if (threadIdx.x == 0 && c) atomicAdd(n, (uint32_t)c);
  }
}

__global__ void __launch_bounds__(kApplyThreads) map_gather_kernel(const MapTable t, bool occupied_only, float thres,
                                                                   uint32_t *pos, unsigned long long *morton,
                                                                   uint32_t *vals) {
  for (uint32_t slot = blockIdx.x; slot < t.cap; slot += gridDim.x) {
    const unsigned long long bk = t.keys[slot];
    if (bk == kMapEmpty) continue;
    for (int half = 0; half < 2; ++half) {
      const uint32_t i = threadIdx.x + half * kApplyThreads;
      if (!exported(t, slot, i, occupied_only, thres)) continue;
      const uint16_t kx = (uint16_t)(((bk & 0xffff) << 3) | (i & 7)),
                     ky = (uint16_t)((((bk >> 16) & 0xffff) << 3) | ((i >> 3) & 7)),
                     kz = (uint16_t)((((bk >> 32) & 0xffff) << 3) | (i >> 6));
      const uint32_t j = atomicAdd(pos, 1u);
      morton[j] = d2pc_map_morton(kx, ky, kz);
      vals[j] = __float_as_uint(t.log_odds[(size_t)slot * 512 + i]);
    }
  }
}

__device__ __forceinline__ void demorton(unsigned long long m, uint16_t k[3]) {
  k[0] = k[1] = k[2] = 0;
  for (int b = 0; b < 16; ++b) {
    k[0] |= (uint16_t)(((m >> (3 * b)) & 1) << b);
    k[1] |= (uint16_t)(((m >> (3 * b + 1)) & 1) << b);
    k[2] |= (uint16_t)(((m >> (3 * b + 2)) & 1) << b);
  }
}

__global__ void __launch_bounds__(kStageThreads) map_write_kernel(const unsigned long long *__restrict__ morton,
                                                                  const uint32_t *__restrict__ vals, uint32_t n,
                                                                  double res, float4 *centres,
                                                                  unsigned long long *keys, float *log_odds) {
  const uint32_t j = blockIdx.x * kStageThreads + threadIdx.x;
  if (j >= n) return;
  uint16_t k[3];
  demorton(morton[j], k);
  if (centres) {
    centres[j] = make_float4(__double2float_rn(d2pc_map_centre(k[0], res)), __double2float_rn(d2pc_map_centre(k[1], res)),
                             __double2float_rn(d2pc_map_centre(k[2], res)), 1.0f);
  } else {
    keys[j] = (unsigned long long)k[0] | ((unsigned long long)k[1] << 16) | ((unsigned long long)k[2] << 32);
    log_odds[j] = __uint_as_float(vals[j]);
  }
}

size_t cub_sort_bytes(uint32_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                  (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)n, 0, 48);
  return bytes;
}

}  // namespace

uint32_t map_table_cap(uint32_t max_bricks) {
  uint32_t cap = 2;
  while (cap < 2ull * max_bricks) cap <<= 1;
  return cap;
}

size_t map_table_bytes(uint32_t max_bricks) {
  const size_t cap = map_table_cap(max_bricks);
  return align_up(cap * 8) + align_up(cap * 512 * 4) + align_up(cap * 16 * 4) + align_up(cap * 512 * 4) +
         align_up(cap * 4) + align_up(cap * 4) + align_up(4 * 4) + align_up(2 * 8);
}

MapTable map_table_carve(uint8_t *base, uint32_t max_bricks) {
  MapTable t;
  t.cap = map_table_cap(max_bricks);
  t.max_bricks = max_bricks;
  const size_t cap = t.cap;
  uint8_t *p = base;
  auto take = [&](size_t bytes) {
    uint8_t *q = p;
    p += align_up(bytes);
    return q;
  };
  t.keys = reinterpret_cast<unsigned long long *>(take(cap * 8));
  t.log_odds = reinterpret_cast<float *>(take(cap * 512 * 4));
  t.known = reinterpret_cast<uint32_t *>(take(cap * 16 * 4));
  t.marks = reinterpret_cast<uint32_t *>(take(cap * 512 * 4));
  t.slot_epoch = reinterpret_cast<uint32_t *>(take(cap * 4));
  t.touched = reinterpret_cast<uint32_t *>(take(cap * 4));
  t.ctr = reinterpret_cast<uint32_t *>(take(4 * 4));
  t.frames = reinterpret_cast<unsigned long long *>(take(2 * 8));
  return t;
}

cudaError_t map_clear(const MapTable &t, bool marks_too, cudaStream_t stream) {
  const size_t cap = t.cap;
  cudaError_t e;
  if ((e = cudaMemsetAsync(t.keys, 0xff, cap * 8, stream)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(t.known, 0, cap * 16 * 4, stream)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(t.ctr, 0, 4 * 4, stream)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(t.frames, 0, 2 * 8, stream)) != cudaSuccess) return e;
  if (marks_too) {
    if ((e = cudaMemsetAsync(t.marks, 0, cap * 512 * 4, stream)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(t.slot_epoch, 0, cap * 4, stream)) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

cudaError_t launch_map_insert(const CloudSrc &in, const MapTable &t, const MapUpdate &u, int sm_count,
                              cudaStream_t stream, int *launches) {
  if (launches) *launches = 0;
  if (in.n_max) {
    map_mark_kernel<<<(in.n_max + kStageThreads - 1) / kStageThreads, kStageThreads, 0, stream>>>(in, t, u);
    if (launches) ++*launches;
  }
  map_apply_kernel<<<sm_count * 8, kApplyThreads, 0, stream>>>(t, u);
  map_finish_kernel<<<1, 1, 0, stream>>>(t);
  const cudaError_t e = cudaGetLastError();
  if (launches && e == cudaSuccess) *launches += 2;
  return e;
}

cudaError_t map_count(const MapTable &t, bool occupied_only, float occ_thres, uint32_t *d_n, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(d_n, 0, 4, stream);
  if (e != cudaSuccess) return e;
  const uint32_t grid = t.cap < 4096 ? t.cap : 4096;
  map_count_kernel<<<grid, kApplyThreads, 0, stream>>>(t, occupied_only, occ_thres, d_n);
  return cudaGetLastError();
}

size_t map_export_temp_bytes(uint32_t n) {
  return 2 * align_up((size_t)n * 8) + 2 * align_up((size_t)n * 4) + cub_sort_bytes(n);
}

cudaError_t map_export(const MapTable &t, bool occupied_only, float occ_thres, double res, uint32_t n, void *temp,
                       uint32_t *d_pos, float4 *centres, unsigned long long *keys, float *log_odds,
                       cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  uint8_t *p = static_cast<uint8_t *>(temp);
  auto *m0 = reinterpret_cast<unsigned long long *>(p);
  auto *m1 = reinterpret_cast<unsigned long long *>(p + align_up((size_t)n * 8));
  auto *v0 = reinterpret_cast<uint32_t *>(p + 2 * align_up((size_t)n * 8));
  auto *v1 = reinterpret_cast<uint32_t *>(p + 2 * align_up((size_t)n * 8) + align_up((size_t)n * 4));
  void *sort_temp = p + 2 * align_up((size_t)n * 8) + 2 * align_up((size_t)n * 4);
  size_t sort_bytes = cub_sort_bytes(n);
  cudaError_t e = cudaMemsetAsync(d_pos, 0, 4, stream);
  if (e != cudaSuccess) return e;
  const uint32_t grid = t.cap < 4096 ? t.cap : 4096;
  map_gather_kernel<<<grid, kApplyThreads, 0, stream>>>(t, occupied_only, occ_thres, d_pos, m0, v0);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = cub::DeviceRadixSort::SortPairs(sort_temp, sort_bytes, m0, m1, v0, v1, (int)n, 0, 48, stream)) !=
      cudaSuccess)
    return e;
  map_write_kernel<<<(n + kStageThreads - 1) / kStageThreads, kStageThreads, 0, stream>>>(m1, v1, n, res, centres,
                                                                                          keys, log_odds);
  return cudaGetLastError();
}

}  // namespace d2pc
