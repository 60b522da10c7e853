// radius_outlier.cu -- pcl::RadiusOutlierRemoval<pcl::PointXYZ> (PCL 1.8 - 1.12, setNegative(false),
// keep_organized false) on the device, batched over frames: the stage that runs behind the filter mode when a
// radius is set, and d2pc_radius_outlier_device.  include/d2pc_b200.h states the recipe; this file finds, for every
// finite point, whether at least min_neighbors + 1 finite points (itself included) lie within the radius:
//
//   1. bounds  cloud_bounds_kernel  per-block min / max of the finite points below count[f] -> partials
//              ror_finish_kernel    one block per frame: partials -> grid (origin, cell size, cells per axis)
//   2. keys    ror_keys_kernel      (frame, linear cell index) -> point index; non-finite points and positions past
//                                   the count get the frame's sentinel cell, which sorts after every real cell
//   3. sort    cub::DeviceRadixSort::SortPairs on all 64 key bits (stable)
//   4. gather  ror_gather_kernel    the points in sorted (cell) order, so that a cell's points are contiguous
//   5. count   ror_count_kernel     one thread per sorted position: for each of the 9 (dy, dz) rows around its cell
//                                   the cells x-1..x+1 are one contiguous key range, found by binary search; rule
//                                   3-4 of the recipe on each point of it, stopping at min_neighbors + 1 -> a flag at
//                                   the point's input position
//   6. output  cloud_stage.cuh's compaction over the flags: kept points copied unchanged in input order, and the
//              per-frame counts
//
// Why the 27 cells around a point hold every neighbour (the margin).  Let r' = max(radius, 2^-64) and let the
// cell size c start at r' * (1 + 2^-10); it only grows.  Take a pair that passes rule 4 with a finite r2 (s <= r2).
//   * s >= fl(dx*dx): the adds of rule 3 round monotonically and add non-negative terms.  So
//     dx^2 <= fl(dx*dx) * (1 + 2^-23) + 2^-150 (round to nearest, the second term for the subnormal range)
//     <= r^2 (1 + 2^-53)(1 + 2^-23) + 2^-150 <= r'^2 (1 + 2^-21), since 2^-150 <= 2^-22 * r'^2.
//   * dx = fl(xi - xj), which is exact in the subnormal range and within a factor (1 - 2^-24) otherwise (an
//     overflow makes s infinite, which fails a finite r2).  So |xi - xj| <= r' (1 + 2^-20).
//   * The cell coordinate is t(x) = fl64(fl64(x - min) * fl64(1 / c)) and the cell floor(t) + 1.  Every axis has at
//     most 2^32 cells (the grid coarsens until it has), so t < 2^32 and the two double roundings of each t move it by
//     less than 2^32 * 2^-52 = 2^-20; 1/c rounds by 2^-53.  Hence t(xi) - t(xj) <= (1 + 2^-20)(1 + 2^-53) /
//     (1 + 2^-10) + 2 * 2^-20 < 1, and the cells of i and j differ by at most one along every axis.
//   * With r2 = inf (radius > 1.3e154) every pair passes, but then c > r > 2 * FLT_MAX exceeds every span and each
//     frame is a single cell.
// The grid is padded by one cell on every side (cells 1..K hold points, 0 and K+1 stay empty), so the ranges of
// the neighbour rows never wrap.  Coarsening (doubling c) keeps all of this true for any finite coordinates; it
// only puts more points into a cell.
//
// Distances are float32 with explicit round-to-nearest intrinsics (no FMA contraction, no fast-math), as the recipe
// requires.  No buffer is read before a kernel of the same launch has written it, so the scratch needs no clearing.
#include "radius_outlier.h"

#include <cub/device/device_radix_sort.cuh>

namespace d2pc {
namespace {

constexpr double kMinCell = 0x1p-64;        // r' = max(radius, kMinCell): see the margin argument above
constexpr double kMargin = 1.0 + 0x1p-10;   // c >= r' * kMargin
constexpr double kMaxAxisCells = 0x1p32;    // per-axis cells, padding included

struct Desc {
  float mn[3];  // per-axis min of the frame's finite points: the low edge of cell 1
  float pad;
  double ic;          // 1 / cell size
  uint64_t dx, dxy;   // cells along x, cells per z layer (padding included)
};

__device__ __forceinline__ bool finite3(const float4 &q) { return isfinite(q.x) && isfinite(q.y) && isfinite(q.z); }

// the bounds pass's predicate: only finite points span the grid
struct Finite {
  __device__ bool operator()(const float4 &q) const { return finite3(q); }
};

// the cell bits of a key with fb frame bits (all set: the frame's sentinel cell), and frame f's bits
__device__ __forceinline__ uint64_t cell_mask(int fb) { return fb ? (1ull << (64 - fb)) - 1 : ~0ull; }
__device__ __forceinline__ uint64_t frame_part(uint32_t f, int fb) { return fb ? (uint64_t)f << (64 - fb) : 0ull; }

// the cell coordinate of a finite coordinate (floor(t) + 1 of the margin argument)
__device__ __forceinline__ uint64_t cell_of(float x, float mn, double ic) {
  return (uint64_t)floor(__dmul_rn(__dsub_rn((double)x, (double)mn), ic)) + 1;
}

// cells per axis D = K + 2 (K holding points, one padding cell on each side) for the frame's bounds v and 1/c;
// false unless every D <= 2^32 and D.x * D.y * D.z < `limit`
__device__ __forceinline__ bool grid_fits(const float (&v)[6], double ic, uint64_t limit, uint64_t (&D)[3]) {
  for (int a = 0; a < 3; ++a) {
    const double t = floor(__dmul_rn(__dsub_rn((double)v[a + 3], (double)v[a]), ic));
    if (!(t + 3.0 <= kMaxAxisCells)) return false;
    D[a] = (uint64_t)t + 3;
  }
  return D[1] <= limit / D[0] && D[2] <= limit / (D[0] * D[1]) && D[0] * D[1] * D[2] < limit;
}

// one block per frame: the grid.  c doubles until grid_fits with limit 2^(64 - frame bits) - 1, so that the
// sentinel's cell index (all bits set) is above every real one.  The bounds are finite floats, so the span is
// finite and a fit comes before c overflows (<= 1100 doublings from 2^-64); should c reach infinity first anyway,
// 1/c = 0 makes the frame a single cell, which is correct for any input.
__global__ void __launch_bounds__(kStageThreads) ror_finish_kernel(const Partial *__restrict__ partials, uint32_t nb,
                                                                   double radius, int fb, Desc *__restrict__ desc) {
  float v[6];
  fold_partials(partials, nb, v);
  if (threadIdx.x != 0) return;
  Desc d = {};
  if (v[0] <= v[3]) {  // at least one finite point (otherwise every key is the sentinel)
    const uint64_t limit = cell_mask(fb);  // the product of the D must stay below the sentinel's index
    uint64_t D[3] = {3, 3, 3};
    double ic = 0.0;
    for (double c = fmax(radius, kMinCell) * kMargin; c <= DBL_MAX; c *= 2.0)
      if (grid_fits(v, 1.0 / c, limit, D)) {
        ic = 1.0 / c;
        break;
      }
    if (ic == 0.0) D[0] = D[1] = D[2] = 3;
    for (int a = 0; a < 3; ++a) d.mn[a] = v[a];
    d.ic = ic;
    d.dx = D[0];
    d.dxy = D[0] * D[1];
  }
  desc[blockIdx.x] = d;
}

__global__ void __launch_bounds__(kStageThreads) ror_keys_kernel(const CloudSrc in, uint32_t total, int fb,
                                                                 const Desc *__restrict__ desc,
                                                                 uint64_t *__restrict__ keys,
                                                                 uint32_t *__restrict__ vals) {
  const uint32_t j = blockIdx.x * kStageThreads + threadIdx.x;
  if (j >= total) return;
  const uint32_t f = j / in.n_max, i = j - f * in.n_max;
  uint64_t cell = cell_mask(fb);
  if (i < frame_count(in, f)) {
    const float4 q = __ldg(frame_points(in, f) + i);
    if (finite3(q)) {
      const Desc d = desc[f];
      cell = cell_of(q.x, d.mn[0], d.ic) + cell_of(q.y, d.mn[1], d.ic) * d.dx + cell_of(q.z, d.mn[2], d.ic) * d.dxy;
    }
  }
  keys[j] = frame_part(f, fb) | cell;
  vals[j] = i;
}

__global__ void __launch_bounds__(kStageThreads) ror_gather_kernel(const CloudSrc in, uint32_t total, int fb,
                                                                   const uint64_t *__restrict__ keys,
                                                                   const uint32_t *__restrict__ vals,
                                                                   float4 *__restrict__ sorted) {
  const uint32_t j = blockIdx.x * kStageThreads + threadIdx.x;
  if (j >= total) return;
  const uint64_t mask = cell_mask(fb);
  if ((keys[j] & mask) == mask) return;  // a sentinel: never read
  sorted[j] = __ldg(frame_points(in, j / in.n_max) + vals[j]);
}

// first position in [lo, hi) whose key is >= k
__device__ __forceinline__ uint32_t lower_bound(const uint64_t *__restrict__ keys, uint32_t lo, uint32_t hi,
                                                uint64_t k) {
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if (keys[mid] < k) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// rows (dy, dz) of the 3 x 3 x 3 block around a cell, the point's own row first: it holds most neighbours, and the
// count stops as soon as it reaches min_neighbors + 1 (the order cannot change a capped count)
__constant__ int8_t kRowDy[9] = {0, -1, 1, 0, -1, 1, 0, -1, 1};
__constant__ int8_t kRowDz[9] = {0, 0, 0, -1, -1, -1, 1, 1, 1};

__global__ void __launch_bounds__(kStageThreads) ror_count_kernel(uint32_t n_max, uint32_t total, int fb, double r2,
                                                                  uint64_t need, const Desc *__restrict__ desc,
                                                                  const uint64_t *__restrict__ keys,
                                                                  const uint32_t *__restrict__ vals,
                                                                  const float4 *__restrict__ sorted,
                                                                  uint8_t *__restrict__ flags) {
  const uint32_t j = blockIdx.x * kStageThreads + threadIdx.x;
  if (j >= total) return;
  const uint32_t f = j / n_max, s0 = f * n_max, s1 = s0 + n_max;
  const uint64_t mask = cell_mask(fb), key = keys[j], cell = key & mask, fp = key & ~mask;
  uint64_t cnt = 0;
  if (cell != mask) {
    const float4 p = sorted[j];
    const Desc d = desc[f];
    for (int r = 0; r < 9 && cnt < need; ++r) {
      // the padding keeps cell +- 1 +- dx +- dxy inside [0, dx * dy * dz): no wrap, no carry into the frame bits
      // (the offsets are added modulo 2^64, which is exact whenever the true result is in range)
      const uint64_t row = cell + (uint64_t)(int64_t)kRowDy[r] * d.dx + (uint64_t)(int64_t)kRowDz[r] * d.dxy;
      const uint32_t lo = lower_bound(keys, s0, s1, fp | (row - 1));
      const uint32_t hi = lower_bound(keys, lo, s1, fp | (row + 2));
      for (uint32_t m = lo; m < hi; ++m) {
        const float4 q = sorted[m];
        const float ex = __fsub_rn(p.x, q.x), ey = __fsub_rn(p.y, q.y), ez = __fsub_rn(p.z, q.z);
        const float s = __fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(ez, ez));
        if ((double)s <= r2 && ++cnt >= need) break;
      }
    }
  }
  flags[s0 + vals[j]] = cnt >= need;  // a sentinel position has cnt 0 < need (need >= 1): dropped
}

// the compaction's keep: the flag at position j (0 or 1)
struct Flagged {
  const uint8_t *flags;
  __device__ uint32_t operator()(const CloudSrc &, uint32_t, uint32_t, uint32_t j) const { return flags[j]; }
};

// every buffer of one launch, carved out of the scratch in this order
struct Layout {
  size_t partials, desc, keys_in, keys_out, vals_in, vals_out, sorted, flags, slot, temp, temp_bytes, total;
};

Layout layout(uint32_t n_frames, uint32_t n_max) {
  const size_t m = (size_t)n_frames * n_max;
  Layout L;
  size_t o = 0;
  L.partials = o, o += align_up((size_t)n_frames * bounds_blocks(n_frames, n_max) * sizeof(Partial));
  L.desc = o, o += align_up((size_t)n_frames * sizeof(Desc));
  L.keys_in = o, o += align_up(m * 8);
  L.keys_out = o, o += align_up(m * 8);
  L.vals_in = o, o += align_up(m * 4);
  L.vals_out = o, o += align_up(m * 4);
  L.sorted = o, o += align_up(m * 16);
  L.flags = o, o += align_up(m);
  L.slot = o, o += align_up((m + 1) * 4);
  size_t sort_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (uint64_t *)nullptr, (uint64_t *)nullptr, (uint32_t *)nullptr,
                                  (uint32_t *)nullptr, (int)m, 0, 64);
  const size_t scan_bytes = compaction_temp_bytes<Flagged>(n_frames, n_max);
  L.temp = o;
  L.temp_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
  o += align_up(L.temp_bytes);
  L.total = o;
  return L;
}

}  // namespace

size_t ror_scratch_bytes(uint32_t n_frames, uint32_t n_max) { return layout(n_frames, n_max).total; }

cudaError_t launch_radius_outlier(const CloudSrc &in, const CloudDst &out, double radius, uint32_t min_neighbors,
                                  void *scratch, cudaStream_t stream, int *launches) {
  if (launches) *launches = 0;
  if (in.n_frames == 0) return cudaSuccess;
  if ((uint64_t)in.n_frames * in.n_max > kCloudMaxPoints) return cudaErrorInvalidValue;  // the caller splits the batch
  if (in.n_max == 0) return cudaMemsetAsync(out.counts, 0, in.n_frames * sizeof(uint32_t), stream);
  const uint32_t total = in.n_frames * in.n_max;
  const int fb = frame_bits(in.n_frames);
  const Layout L = layout(in.n_frames, in.n_max);
  uint8_t *base = static_cast<uint8_t *>(scratch);
  Partial *partials = reinterpret_cast<Partial *>(base + L.partials);
  Desc *desc = reinterpret_cast<Desc *>(base + L.desc);
  uint64_t *keys_in = reinterpret_cast<uint64_t *>(base + L.keys_in);
  uint64_t *keys_out = reinterpret_cast<uint64_t *>(base + L.keys_out);
  uint32_t *vals_in = reinterpret_cast<uint32_t *>(base + L.vals_in);
  uint32_t *vals_out = reinterpret_cast<uint32_t *>(base + L.vals_out);
  float4 *sorted = reinterpret_cast<float4 *>(base + L.sorted);
  uint8_t *flags = base + L.flags;
  uint32_t *slot = reinterpret_cast<uint32_t *>(base + L.slot);
  void *temp = base + L.temp;

  // every launch is checked before anything that reads its output is queued
  const uint32_t nb = bounds_blocks(in.n_frames, in.n_max);
  cloud_bounds_kernel<<<nb * in.n_frames, kStageThreads, 0, stream>>>(in, nb, Finite{}, partials);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  ror_finish_kernel<<<in.n_frames, kStageThreads, 0, stream>>>(partials, nb, radius, fb, desc);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  const uint32_t grid = (total + kStageThreads - 1) / kStageThreads;
  ror_keys_kernel<<<grid, kStageThreads, 0, stream>>>(in, total, fb, desc, keys_in, vals_in);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  size_t tb = L.temp_bytes;
  e = cub::DeviceRadixSort::SortPairs(temp, tb, keys_in, keys_out, vals_in, vals_out, (int)total, 0, 64, stream);
  if (e != cudaSuccess) return e;
  ror_gather_kernel<<<grid, kStageThreads, 0, stream>>>(in, total, fb, keys_out, vals_out, sorted);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  ror_count_kernel<<<grid, kStageThreads, 0, stream>>>(in.n_max, total, fb, radius * radius,
                                                       (uint64_t)min_neighbors + 1, desc, keys_out, vals_out, sorted,
                                                       flags);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  e = launch_compaction(in, Flagged{flags}, slot, temp, L.temp_bytes, out, stream);
  // six kernels of this file and cloud_stage.cuh, the sort and the scan (each CUB call counted once)
  if (launches && e == cudaSuccess) *launches = 8;
  return e;
}

}  // namespace d2pc
