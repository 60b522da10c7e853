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
// The export sorts the known voxels by Morton code (map_sort); the octomap serialization below builds the tree on it,
// and the projected 2-D map after it reads each voxel's leaf level from the same front.
#include <cstring>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

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

cudaError_t map_sort(const MapTable &t, bool occupied_only, float occ_thres, uint32_t n, void *temp, uint32_t *d_pos,
                     const unsigned long long **morton, const uint32_t **vals, cudaStream_t stream) {
  uint8_t *p = static_cast<uint8_t *>(temp);
  auto *m0 = reinterpret_cast<unsigned long long *>(p);
  auto *m1 = reinterpret_cast<unsigned long long *>(p + align_up((size_t)n * 8));
  auto *v0 = reinterpret_cast<uint32_t *>(p + 2 * align_up((size_t)n * 8));
  auto *v1 = reinterpret_cast<uint32_t *>(p + 2 * align_up((size_t)n * 8) + align_up((size_t)n * 4));
  void *sort_temp = p + 2 * align_up((size_t)n * 8) + 2 * align_up((size_t)n * 4);
  size_t sort_bytes = cub_sort_bytes(n);
  *morton = m1;
  *vals = v1;
  cudaError_t e = cudaMemsetAsync(d_pos, 0, 4, stream);
  if (e != cudaSuccess) return e;
  const uint32_t grid = t.cap < 4096 ? t.cap : 4096;
  map_gather_kernel<<<grid, kApplyThreads, 0, stream>>>(t, occupied_only, occ_thres, d_pos, m0, v0);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  return cub::DeviceRadixSort::SortPairs(sort_temp, sort_bytes, m0, m1, v0, v1, (int)n, 0, 48, stream);
}

cudaError_t map_export(const MapTable &t, bool occupied_only, float occ_thres, double res, uint32_t n, void *temp,
                       uint32_t *d_pos, float4 *centres, unsigned long long *keys, float *log_odds,
                       cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const unsigned long long *m;
  const uint32_t *v;
  cudaError_t e = map_sort(t, occupied_only, occ_thres, n, temp, d_pos, &m, &v, stream);
  if (e != cudaSuccess) return e;
  map_write_kernel<<<(n + kStageThreads - 1) / kStageThreads, kStageThreads, 0, stream>>>(m, v, n, res, centres,
                                                                                          keys, log_odds);
  return cudaGetLastError();
}

// ---- octomap_msgs/Octomap serialization (the recipe is in include/d2pc_b200.h)
//
// From the known voxels sorted by Morton code (map_sort), with n voxels, s_i the first level at which voxel i starts
// a node (0 for i = 0, else 1 + the leading equal 3-bit digits of m_i and m_{i-1}) and lambda_i the shallowest leaf
// level on its path, voxel i writes the nodes of levels s_i .. lambda_i (full) or s_i .. lambda_i - 1 (binary, inner
// nodes only), none when lambda_i < s_i (it lies inside a leaf an earlier voxel wrote).  Node (L, i), started by voxel
// i, is record off_i + L - s_i in either format, so a voxel's records are consecutive and pre-order is voxel order.
//   octo_flags  runs d_i = (v_i != v_{i-1}) and s_i
//   (scan)      D = inclusive sum of d: v is constant on [a, b] iff D_a == D_b
//   octo_levels lambda_i: node (L, i) is full when the codes at both ends of its 8^(16-L) aligned range are present,
//               and a leaf when full and constant; leaf(L) implies leaf(L + 1), so lambda is found from level 16 up.
//               Writes the record count of the format
//   (scan)      off over n + 1 counts: off_n is the total, the one value the host waits for
//   octo_link   per writing voxel: the parent record of its first node (a binary search for the parent's first
//               voxel unless i starts the parent too), then each of its nodes ORs its child bit (full) or its 2-bit
//               code (binary) into its parent's record in the output; the binary stream is complete here
//   octo_max    full only, levels 16 .. 1: each node of the level atomicMax'es its value into its parent's
//   octo_emit   full only: the 4 value bytes of every record
namespace {

constexpr int kOctoThreads = 256;

__device__ __forceinline__ uint32_t ordered(uint32_t f) { return f ^ ((f >> 31) ? 0xffffffffu : 0x80000000u); }
__device__ __forceinline__ uint32_t unordered(uint32_t o) { return o ^ ((o >> 31) ? 0x80000000u : 0xffffffffu); }
__device__ __forceinline__ uint32_t level_of(uint16_t sl) { return sl & 0xff; }      // s
__device__ __forceinline__ uint32_t leaf_of(uint16_t sl) { return sl >> 8; }         // lambda
__device__ __forceinline__ uint32_t digit(unsigned long long m, uint32_t level) {   // child index of node (level)
  return (uint32_t)(m >> (3 * (16 - level))) & 7u;
}

__global__ void __launch_bounds__(kOctoThreads) octo_flags_kernel(const unsigned long long *__restrict__ m,
                                                                  const uint32_t *__restrict__ v, uint32_t n,
                                                                  uint32_t *d, uint16_t *sl) {
  const uint32_t i = blockIdx.x * kOctoThreads + threadIdx.x;
  if (i >= n) return;
  uint32_t s = 0, diff = 0;
  if (i > 0) {
    const int h = 63 - __clzll((long long)(m[i] ^ m[i - 1]));  // codes are distinct
    s = 16 - h / 3;
    diff = v[i] != v[i - 1];
  }
  d[i] = diff;
  sl[i] = (uint16_t)s;
}

__global__ void __launch_bounds__(kOctoThreads) octo_levels_kernel(const unsigned long long *__restrict__ m,
                                                                   const uint32_t *__restrict__ D, uint32_t n,
                                                                   bool binary, uint16_t *sl,
                                                                   unsigned long long *cnt) {
  const uint32_t i = blockIdx.x * kOctoThreads + threadIdx.x;
  if (i > n) return;
  if (i == n) {
    cnt[n] = 0;
    return;
  }
  const unsigned long long mi = m[i];
  uint32_t lam = 16;
  for (int L = 15; L >= 0; --L) {
    const unsigned long long size = 1ull << (3 * (16 - L)), off = mi & (size - 1);
    if (size > n || off > i) break;
    const unsigned long long a = i - off, b = a + size - 1;
    if (b >= n || m[a] != mi - off || m[b] != mi - off + size - 1 || D[a] != D[b]) break;
    lam = (uint32_t)L;
  }
  const uint32_t s = level_of(sl[i]);
  sl[i] = (uint16_t)(s | (lam << 8));
  cnt[i] = lam < s ? 0 : lam - s + (binary ? 0 : 1);
}

// The record of node (level, voxel p), p its first voxel.
__device__ __forceinline__ unsigned long long record(const unsigned long long *off, const uint16_t *sl, uint32_t p,
                                                     uint32_t level) {
  return off[p] + level - level_of(sl[p]);
}

// ORs `bits` into byte `at` of the output (the word that holds it: the other bytes are left as they are).
__device__ __forceinline__ void or_byte(uint8_t *out, unsigned long long at, uint32_t bits) {
  atomicOr(reinterpret_cast<uint32_t *>(out + (at & ~3ull)), bits << (8 * (at & 3)));
}

__global__ void __launch_bounds__(kOctoThreads) octo_link_kernel(const unsigned long long *__restrict__ m,
                                                                 const uint32_t *__restrict__ v,
                                                                 const uint16_t *__restrict__ sl,
                                                                 const unsigned long long *__restrict__ off,
                                                                 uint32_t n, bool binary, float occ_thres,
                                                                 unsigned long long *up, uint8_t *out) {
  const uint32_t i = blockIdx.x * kOctoThreads + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = level_of(sl[i]), lam = leaf_of(sl[i]);
  if (lam < s) return;
  const unsigned long long mi = m[i], r0 = off[i];
  if (s > 0) {
    // the parent (level s - 1) started at an earlier voxel: the first one whose code has the parent's prefix
    const uint32_t P = s - 1;
    const unsigned long long base = mi & ~((1ull << (3 * (16 - P))) - 1);
    uint32_t lo = (mi - base) > i ? 0 : (uint32_t)(i - (mi - base)), hi = i - 1;
    while (lo < hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (m[mid] < base) lo = mid + 1;
      else hi = mid;
    }
    up[i] = record(off, sl, lo, P);
  }
  const float val = __uint_as_float(v[i]);
  for (uint32_t L = s > 0 ? s : 1; L <= lam; ++L) {
    const unsigned long long parent = L == s ? up[i] : r0 + (L - 1 - s);
    const uint32_t c = digit(mi, L);
    if (binary) {
      const uint32_t code = L < lam ? 3u : (val >= occ_thres ? 2u : 1u);
      const uint32_t bits = code << (2 * c);  // a little-endian uint16: children 0-3 in byte 0, 4-7 in byte 1
      if (bits & 0xff) or_byte(out, 2 * parent, bits & 0xff);
      if (bits >> 8) or_byte(out, 2 * parent + 1, bits >> 8);
    } else {
      or_byte(out, 5 * parent + 4, 1u << c);
    }
  }
}

// level L's nodes into their parents' values (vmax holds ordered floats, 0 below every value)
__global__ void __launch_bounds__(kOctoThreads) octo_max_kernel(const uint32_t *__restrict__ v,
                                                                const uint16_t *__restrict__ sl,
                                                                const unsigned long long *__restrict__ off,
                                                                const unsigned long long *__restrict__ up, uint32_t n,
                                                                uint32_t L, uint32_t *vmax) {
  const uint32_t i = blockIdx.x * kOctoThreads + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = level_of(sl[i]), lam = leaf_of(sl[i]);
  if (L < s || L > lam) return;
  const unsigned long long r = off[i] + (L - s);
  const uint32_t val = L == lam ? ordered(v[i]) : vmax[r];
  atomicMax(vmax + (L == s ? up[i] : r - 1), val);
}

__global__ void __launch_bounds__(kOctoThreads) octo_emit_kernel(const uint32_t *__restrict__ v,
                                                                 const uint16_t *__restrict__ sl,
                                                                 const unsigned long long *__restrict__ off,
                                                                 const uint32_t *__restrict__ vmax, uint32_t n,
                                                                 uint8_t *out) {
  const uint32_t i = blockIdx.x * kOctoThreads + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = level_of(sl[i]), lam = leaf_of(sl[i]);
  for (uint32_t L = s; L <= lam; ++L) {
    const unsigned long long r = off[i] + (L - s);
    const uint32_t f = L == lam ? v[i] : unordered(vmax[r]);
    uint8_t *p = out + 5 * r;
    p[0] = (uint8_t)f, p[1] = (uint8_t)(f >> 8), p[2] = (uint8_t)(f >> 16), p[3] = (uint8_t)(f >> 24);
  }
}

size_t cub_sum_bytes(uint32_t n) {
  size_t a = 0, b = 0;
  cub::DeviceScan::InclusiveSum(nullptr, a, (const uint32_t *)nullptr, (uint32_t *)nullptr, (int)n);
  cub::DeviceScan::ExclusiveSum(nullptr, b, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                (int)n + 1);
  return a > b ? a : b;
}

// the parts of the octomap scratch behind map_sort's
struct OctoTemp {
  uint32_t *d, *D;
  uint16_t *sl;
  unsigned long long *cnt, *off, *up;
  void *scan;
  size_t scan_bytes;
};
OctoTemp octo_temp(void *temp, uint32_t n) {
  uint8_t *p = static_cast<uint8_t *>(temp) + align_up(map_export_temp_bytes(n));  // CUB's part is not aligned
  OctoTemp o;
  auto take = [&](size_t bytes) {
    uint8_t *q = p;
    p += align_up(bytes);
    return q;
  };
  o.d = reinterpret_cast<uint32_t *>(take((size_t)n * 4));
  o.D = reinterpret_cast<uint32_t *>(take((size_t)n * 4));
  o.sl = reinterpret_cast<uint16_t *>(take((size_t)n * 2));
  o.cnt = reinterpret_cast<unsigned long long *>(take(((size_t)n + 1) * 8));
  o.off = reinterpret_cast<unsigned long long *>(take(((size_t)n + 1) * 8));
  o.up = o.cnt;  // the counts are dead once scanned
  o.scan_bytes = cub_sum_bytes(n);
  o.scan = take(o.scan_bytes);
  return o;
}

// map_sort's output inside temp
void sorted_of(const void *temp, uint32_t n, const unsigned long long **m, const uint32_t **v) {
  const uint8_t *p = static_cast<const uint8_t *>(temp);
  *m = reinterpret_cast<const unsigned long long *>(p + align_up((size_t)n * 8));
  *v = reinterpret_cast<const uint32_t *>(p + 2 * align_up((size_t)n * 8) + align_up((size_t)n * 4));
}

// The front the octomap export and the projected map share: the voxels sorted (map_sort), then each voxel's first
// and leaf level in o.sl and the record count of `binary` in o.cnt (octo_flags, the inclusive scan, octo_levels).
cudaError_t octo_front(const MapTable &t, uint32_t n, bool binary, void *temp, uint32_t *d_pos, OctoTemp o,
                       cudaStream_t stream) {
  const unsigned long long *m;
  const uint32_t *v;
  cudaError_t e = map_sort(t, false, 0.0f, n, temp, d_pos, &m, &v, stream);
  if (e != cudaSuccess) return e;
  const uint32_t grid = (n + kOctoThreads - 1) / kOctoThreads, grid1 = n / kOctoThreads + 1;
  octo_flags_kernel<<<grid, kOctoThreads, 0, stream>>>(m, v, n, o.d, o.sl);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = cub::DeviceScan::InclusiveSum(o.scan, o.scan_bytes, o.d, o.D, (int)n, stream)) != cudaSuccess) return e;
  octo_levels_kernel<<<grid1, kOctoThreads, 0, stream>>>(m, o.D, n, binary, o.sl, o.cnt);
  return cudaGetLastError();
}

}  // namespace

size_t octomap_temp_bytes(uint32_t n) {
  return align_up(map_export_temp_bytes(n)) + 2 * align_up((size_t)n * 4) + align_up((size_t)n * 2) +
         2 * align_up(((size_t)n + 1) * 8) + align_up(cub_sum_bytes(n));
}

cudaError_t octomap_plan(const MapTable &t, uint32_t n, bool binary, void *temp, uint32_t *d_pos,
                         unsigned long long *records, cudaStream_t stream) {
  OctoTemp o = octo_temp(temp, n);
  cudaError_t e = octo_front(t, n, binary, temp, d_pos, o, stream);
  if (e != cudaSuccess) return e;
  if ((e = cub::DeviceScan::ExclusiveSum(o.scan, o.scan_bytes, o.cnt, o.off, (int)n + 1, stream)) != cudaSuccess)
    return e;
  return cudaMemcpyAsync(records, o.off + n, 8, cudaMemcpyDeviceToHost, stream);
}

size_t octomap_out_bytes(unsigned long long records, bool binary) {
  return binary ? align_up(records * 2 + 4) : align_up(records * 5 + 4) + align_up(records * 4);
}

cudaError_t octomap_emit(const MapTable &t, uint32_t n, bool binary, float occ_thres, void *temp,
                         unsigned long long records, uint8_t *out, cudaStream_t stream) {
  const OctoTemp o = octo_temp(temp, n);
  const unsigned long long *m;
  const uint32_t *v;
  sorted_of(temp, n, &m, &v);
  const size_t bytes = binary ? records * 2 : records * 5;
  uint32_t *vmax = binary ? nullptr : reinterpret_cast<uint32_t *>(out + align_up(bytes + 4));
  cudaError_t e = cudaMemsetAsync(out, 0, bytes, stream);
  if (e != cudaSuccess) return e;
  if (vmax && (e = cudaMemsetAsync(vmax, 0, records * 4, stream)) != cudaSuccess) return e;
  const uint32_t grid = (n + kOctoThreads - 1) / kOctoThreads;
  octo_link_kernel<<<grid, kOctoThreads, 0, stream>>>(m, v, o.sl, o.off, n, binary, occ_thres, o.up, out);
  if (!binary) {
    for (uint32_t L = 16; L >= 1; --L)
      octo_max_kernel<<<grid, kOctoThreads, 0, stream>>>(v, o.sl, o.off, o.up, n, L, vmax);
    octo_emit_kernel<<<grid, kOctoThreads, 0, stream>>>(v, o.sl, o.off, vmax, n, out);
  }
  return cudaGetLastError();
}

// ---- octomap_server's projected 2-D map, nav_msgs/OccupancyGrid (the recipe is in include/d2pc_b200.h)
//
// On the voxels octo_front sorted and levelled, one thread per voxel with its leaf level lambda_i.  Every voxel of a
// leaf has the leaf's level and value, and the leaf's voxels fill it, so what each voxel does with its leaf's extent,
// height test and value over its own column is, over all of them, what octomap does with the leaf.
//   proj_extent  the leaf's lo and hi per axis, reduced over the warp and the block, then one atomicMin per block
//                into 6 words: ordered encodings of the minima, complemented ones of the maxima (so one 0xff memset
//                starts all six).  The host reads them (the call's one extra wait) and sizes the grid
//   proj_fill    a leaf that passes the height test ORs 1 (free) or 2 (occupied) into its voxel's cell byte; the
//                byte is read first, as most voxels share their column with others
//   proj_emit    the codes into OccupancyGrid values: 2 or 3 -> 100, 1 -> 0, 0 -> -1
namespace {

constexpr int kProjThreads = 256;

__device__ __forceinline__ unsigned long long ordered64(double d) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(d);
  return (b >> 63) ? ~b : b | 0x8000000000000000ull;
}
double unordered64(unsigned long long o) {
  const unsigned long long b = (o >> 63) ? o & 0x7fffffffffffffffull : ~o;
  double d;
  memcpy(&d, &b, 8);
  return d;
}
__device__ __forceinline__ unsigned long long umin64(unsigned long long a, unsigned long long b) { return b < a ? b : a; }

__global__ void __launch_bounds__(kProjThreads) proj_extent_kernel(const unsigned long long *__restrict__ m,
                                                                   const uint16_t *__restrict__ sl, uint32_t n,
                                                                   double res, unsigned long long *ext) {
  const uint32_t i = blockIdx.x * kProjThreads + threadIdx.x;
  unsigned long long e[6];
  for (int a = 0; a < 6; ++a) e[a] = ~0ull;
  if (i < n) {
    uint16_t k[3];
    demorton(m[i], k);
    const uint32_t lam = leaf_of(sl[i]);
    // calcMinMax: lo = c - size / 2, hi = lo + size
    const double size = d2pc_map_node_size(lam, res), half = __ddiv_rn(size, 2.0);
    for (int a = 0; a < 3; ++a) {
      const double lo = __dsub_rn(d2pc_map_node_centre(k[a], lam, res), half);
      e[a] = ordered64(lo);
      e[3 + a] = ~ordered64(__dadd_rn(lo, size));
    }
  }
  __shared__ unsigned long long part[6][kProjThreads / 32];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int a = 0; a < 6; ++a) {
    for (int s = 16; s > 0; s >>= 1) e[a] = umin64(e[a], __shfl_xor_sync(0xffffffffu, e[a], s));
    if (lane == 0) part[a][warp] = e[a];
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    unsigned long long r = part[threadIdx.x][0];
    for (int w = 1; w < kProjThreads / 32; ++w) r = umin64(r, part[threadIdx.x][w]);
    if (r != ~0ull) atomicMin(ext + threadIdx.x, r);
  }
}

__global__ void __launch_bounds__(kProjThreads) proj_fill_kernel(const unsigned long long *__restrict__ m,
                                                                 const uint32_t *__restrict__ v,
                                                                 const uint16_t *__restrict__ sl, uint32_t n,
                                                                 double res, double min_z, double max_z,
                                                                 float occ_thres, const ProjGrid g, uint8_t *cells) {
  const uint32_t i = blockIdx.x * kProjThreads + threadIdx.x;
  if (i >= n) return;
  uint16_t k[3];
  demorton(m[i], k);
  const uint32_t lam = leaf_of(sl[i]);
  const double half = __ddiv_rn(d2pc_map_node_size(lam, res), 2.0), cz = d2pc_map_node_centre(k[2], lam, res);
  if (!(__dadd_rn(cz, half) > min_z && __dsub_rn(cz, half) < max_z)) return;
  const uint32_t code = __uint_as_float(v[i]) >= occ_thres ? 2u : 1u;
  // the padded min key is at most the least key of the map on each axis and the padded max at least the largest
  // (both come within one key of a leaf's face), so the cell is inside the grid
  const unsigned long long at =
      (unsigned long long)(k[1] - g.min_key[1]) * g.width + (unsigned long long)(k[0] - g.min_key[0]);
  if (!(cells[at] & code)) or_byte(cells, at, code);
}

__global__ void __launch_bounds__(kProjThreads) proj_emit_kernel(uint4 *cells, unsigned long long vecs) {
  for (unsigned long long j = (unsigned long long)blockIdx.x * kProjThreads + threadIdx.x; j < vecs;
       j += (unsigned long long)gridDim.x * kProjThreads) {
    uint4 c = cells[j];
    uint32_t *w = &c.x;
    for (int q = 0; q < 4; ++q) {
      uint32_t out = 0;
      for (int b = 0; b < 4; ++b) {
        const uint32_t code = (w[q] >> (8 * b)) & 3u;
        out |= (code & 2u ? 100u : code ? 0u : 0xffu) << (8 * b);
      }
      w[q] = out;
    }
    cells[j] = c;
  }
}

}  // namespace

cudaError_t projmap_extent(const MapTable &t, uint32_t n, double res, void *temp, uint32_t *d_pos,
                           unsigned long long *d_ext, unsigned long long *h_ext, cudaStream_t stream) {
  const OctoTemp o = octo_temp(temp, n);
  // the front also writes the binary format's record counts into o.cnt; the projection needs only the leaf levels
  cudaError_t e = octo_front(t, n, true, temp, d_pos, o, stream);
  if (e != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(d_ext, 0xff, 6 * 8, stream)) != cudaSuccess) return e;
  const unsigned long long *m;
  const uint32_t *v;
  sorted_of(temp, n, &m, &v);
  proj_extent_kernel<<<(n + kProjThreads - 1) / kProjThreads, kProjThreads, 0, stream>>>(m, o.sl, n, res, d_ext);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  return cudaMemcpyAsync(h_ext, d_ext, 6 * 8, cudaMemcpyDeviceToHost, stream);
}

bool projmap_grid(const unsigned long long ext[6], double res, double min_x_size, double min_y_size, ProjGrid *g) {
  double mn[3], mx[3];
  for (int a = 0; a < 3; ++a) mn[a] = unordered64(ext[a]), mx[a] = unordered64(~ext[3 + a]);
  // the padding: std::min(a, b) is (b < a) ? b : a, std::max(a, b) is (a < b) ? b : a
  const double half[2] = {0.5 * min_x_size, 0.5 * min_y_size};
  for (int a = 0; a < 2; ++a) {
    if (-half[a] < mn[a]) mn[a] = -half[a];
    if (mx[a] < half[a]) mx[a] = half[a];
  }
  // float point3d corners, coordToKeyChecked on all three axes
  const double rf = 1.0 / res;
  uint16_t lo[3], hi[3];
  if (!d2pc_map_key3(rf, (float)mn[0], (float)mn[1], (float)mn[2], lo) ||
      !d2pc_map_key3(rf, (float)mx[0], (float)mx[1], (float)mx[2], hi))
    return false;
  for (int a = 0; a < 2; ++a) {
    g->min_key[a] = lo[a];
    g->origin[a] = (double)(float)d2pc_map_centre(lo[a], res) - res * 0.5;
  }
  g->width = (uint32_t)(hi[0] - lo[0]) + 1u;
  g->height = (uint32_t)(hi[1] - lo[1]) + 1u;
  return true;
}

size_t projmap_cells_bytes(const ProjGrid &g) { return ((size_t)g.width * g.height + 15) & ~(size_t)15; }

cudaError_t projmap_fill(const MapTable &t, uint32_t n, double res, double min_z, double max_z, float occ_thres,
                         void *temp, const ProjGrid &g, uint8_t *cells, cudaStream_t stream) {
  const size_t bytes = projmap_cells_bytes(g);
  cudaError_t e = cudaMemsetAsync(cells, 0, bytes, stream);
  if (e != cudaSuccess) return e;
  const OctoTemp o = octo_temp(temp, n);
  const unsigned long long *m;
  const uint32_t *v;
  sorted_of(temp, n, &m, &v);
  proj_fill_kernel<<<(n + kProjThreads - 1) / kProjThreads, kProjThreads, 0, stream>>>(m, v, o.sl, n, res, min_z,
                                                                                        max_z, occ_thres, g, cells);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  const unsigned long long vecs = bytes / 16, want = (vecs + kProjThreads - 1) / kProjThreads;
  const uint32_t grid = (uint32_t)(want < 65536 ? want : 65536);
  proj_emit_kernel<<<grid, kProjThreads, 0, stream>>>(reinterpret_cast<uint4 *>(cells), vecs);
  return cudaGetLastError();
}

}  // namespace d2pc
