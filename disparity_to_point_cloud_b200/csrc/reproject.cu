// reproject.cu -- the disparity callback's reprojection + crop + pack on sm_100a.
//
// Replaces, in ONE pass over HBM (4 B read + 16 B written per kept pixel):
//   cv::reprojectImageTo3D(real_disparity, image3D, Q_)   src/disparity_to_point_cloud.cpp:63-64
//   the 40-pixel border crop loop + pcl::PointXYZ push_back   :69-76
//   pcl::toROSMsg's memcpy into PointCloud2.data              :84-85
// and, for the mono8 entry, Mat::convertTo(CV_32FC1, 1/8)     :60-61.
//
// CROP kernel (reference-exact filter: output offsets are closed form)
//   work unit = 128 crop columns x RB crop rows, one warp per unit, one unit per warp (the CTA scheduler balances).
//   Per row: each lane issues one 16-byte streaming load (4 disparities), the
//   warp transposes through 512 B of shared memory so that lane L then owns
//   pixels L, L+32, L+64, L+96 -- which makes every one of the four 16-byte
//   point stores of the warp a contiguous 512-byte burst.  Column constants
//   (X) live in registers for the whole unit, row constants (Y) are computed
//   by one lane each and broadcast by shuffle; Q sits in the kernel parameter
//   (constant) bank.  Each warp prefetches into L2 (cp.async.bulk.prefetch.L2)
//   the unit a warp launched a fraction of a wave later will read.
//
// CROP_FINITE kernels (extension: drop non-finite points, keep row-major order)
//   band kernel (default for the stereoRectify form of Q): a CTA owns whole crop rows; TMA bulk row loads,
//   survivors counted from the disparity alone (four units per REDUX), block scan, ONE decoupled look-back per
//   band over 64-bit {epoch,flag,value} descriptors, survivors reprojected and stored at offset + ballot rank.
//   park kernel (any other Q, FAST mode): 32-unit tiles, points parked in shared memory because validity is only
//   known after the arithmetic, same look-back.
//   (Round 1 also carried a classify-first tile kernel, a two-pass count / scan / store variant and a
//   warp-specialised TMA pipeline kernel: all correct, all 1.3-2x slower than the band kernel; removed in round 2,
//   their measurements are kept in DESIGN.md.)
#include "reproject.h"

#include <cuda.h>
#include <cudaTypedefs.h>

#include <algorithm>
#include <cmath>

#include "reproject_math.cuh"

namespace d2pc {

namespace {

constexpr int kWarpsPerCta = 4;
constexpr int kThreads = kWarpsPerCta * 32;
constexpr int kSegCols = 128;  // crop columns per warp-row: 32 lanes x 4

// n / d for n < 2^31 as one 32 x 32 -> 64 multiply and a shift (d fixed per launch; the hardware has no integer
// divide, and a unit decode with four of them was a tenth of the CROP kernel's instructions).
// magic = ceil(2^(32+s) / d), s = ceil(log2 d) - 1: magic < 2^32, and e = magic * d - 2^(32+s) < d gives an exact
// quotient while n * e < 2^(32+s), i.e. for every n < 2^31.
struct FastDiv {
  uint32_t magic, shift;  // shift == 0: d == 1
};
static FastDiv make_fastdiv(uint32_t d) {
  FastDiv f{0u, 0u};
  if (d <= 1) return f;
  uint32_t s = 0;
  while ((1ull << (s + 1)) < d) ++s;  // ceil(log2 d) - 1
  f.shift = 32 + s;
  f.magic = (uint32_t)(((1ull << f.shift) + d - 1) / d);
  return f;
}
__device__ __forceinline__ uint32_t fastdiv(uint32_t n, FastDiv f) {
  return f.shift == 0u ? n : (uint32_t)(((unsigned long long)n * f.magic) >> f.shift);
}

struct ReprojArgs {
  CUtensorMap tmap;  // CROP kernel, TMA form: crop columns x crop rows x frames of the input
  bool tma;
  const uint8_t *in;
  size_t step, frame_stride;
  float4 *out;
  size_t out_frame_stride;  // in points
  uint32_t *counts;
  int n_frames, width, height, border, cw, ch;
  int rows_per_unit, n_seg, n_rb;
  uint32_t units_per_frame, total_units;
  FastDiv div_upf, div_nseg;  // CROP kernel: unit -> (frame, row block, segment) without integer divisions
  float scale;
  // compaction
  unsigned long long *tile_desc;
  uint32_t *ticket;
  uint32_t epoch, tiles_per_frame;
  const double *xtab, *ytab;  // (double)(float)(u + q03), (double)(float)(v + q13)
  uint32_t d_sure_bits;       // float bits of the smallest |d| whose point is certainly finite (rect0 compaction)
  int band_rows, cw_pad, band_groups, group_rows;  // band kernel geometry
  int prefetch_dist;          // band kernel: L2 prefetch distance in tiles (0 = off)
  QParams Q;
};

// M: Markstein quotients.  Z: kMathRect0 for a calibration whose principal point column is an image column (X is
// exactly 0 there): zero numerators stay on the straight-line path instead of taking the exact function -- 4-25 %
// faster for such a Q, 2-4 % slower for any other (a few more instructions per pixel), hence chosen on the host.
// Probe: no arithmetic, the CROP kernels store {d, d, d, 1} -- the traffic of the reprojection alone (test hook that
// measures the memory ceiling of the CROP kernels' access pattern).
enum { kMathRect0 = 0, kMathRectW = 1, kMathGeneric = 2, kMathFast = 3, kMathRect0M = 4, kMathRect0Z = 5, kMathProbe = 6 };
#define D2PC_IS_RECT(m) ((m) == kMathRect0 || (m) == kMathRectW || (m) == kMathRect0M || (m) == kMathRect0Z)
#define D2PC_IS_GUARD(m) ((m) == kMathRect0 || (m) == kMathRect0Z)

__device__ __forceinline__ float4 ld_stream_f4(const float4 *p) {
  float4 v;
  asm volatile("ld.global.cs.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream_f4(float4 *p, const float4 &v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ void st_stream_f4_if(float4 *p, const float4 &v, bool pred) {  // predicated, no branch
  asm volatile(
      "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %5, 0;\n\t@q st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};\n\t}" ::"l"(p),
      "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"((int)pred)
      : "memory");
}

// One pixel slot of a warp goes to out[pos + rank]: rank by ballot + popc, with the (very common) all-kept and
// none-kept slots short-circuited by a warp-uniform test.  Returns pos advanced by the number of points stored.
__device__ __forceinline__ uint32_t store_ranked(float4 *out, uint32_t pos, const float4 &p, bool keep, int lane,
                                                 uint32_t lt_mask) {
  const uint32_t bal = __ballot_sync(0xffffffffu, keep);
  if (bal == 0xffffffffu) {
    __stcs(out + (pos + (uint32_t)lane), p);
    return pos + 32u;
  }
  if (bal == 0u) return pos;
  if (keep) __stcs(out + (pos + (uint32_t)__popc(bal & lt_mask)), p);
  return pos + (uint32_t)__popc(bal);
}

// Minimal-instruction form: no short-circuits, the lane mask comes from the special register.
__device__ __forceinline__ uint32_t store_ranked_tight(float4 *out, uint32_t pos, const float4 &p, bool keep) {
  uint32_t lt;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt));
  const uint32_t bal = __ballot_sync(0xffffffffu, keep);
  unsigned long long addr;  // out + (pos + rank) * 16 in one IMAD.WIDE
  asm("mad.wide.u32 %0, %1, 16, %2;" : "=l"(addr) : "r"(pos + (uint32_t)__popc(bal & lt)), "l"(out));
  if (keep) __stcs(reinterpret_cast<float4 *>(addr), p);
  return pos + (uint32_t)__popc(bal);
}
// |x|, |y|, |z| all below infinity (false for NaN): three chained float compares.
__device__ __forceinline__ bool point_is_finite_fast(const float4 &p) {
  const float inf = __uint_as_float(0x7f800000u);
  return fabsf(p.x) < inf && fabsf(p.y) < inf && fabsf(p.z) < inf;
}

// src/disparity_to_point_cloud.cpp:61 -- convertTo(CV_32FC1, 1/8): float(src)*alpha + 0
__device__ __forceinline__ float u8_to_disp(uint32_t b, float scale) {
  return __fadd_rn(__fmul_rn((float)b, scale), 0.0f);
}

template <typename InT>
__device__ __forceinline__ float4 load4(const uint8_t *row, int col, float scale);
template <>
__device__ __forceinline__ float4 load4<float>(const uint8_t *row, int col, float) {
  return ld_stream_f4(reinterpret_cast<const float4 *>(row + (size_t)col * 4));
}
template <>
__device__ __forceinline__ float4 load4<uint8_t>(const uint8_t *row, int col, float scale) {
  const uint32_t w = __ldcs(reinterpret_cast<const uint32_t *>(row + col));
  return make_float4(u8_to_disp(w & 0xff, scale), u8_to_disp((w >> 8) & 0xff, scale),
                     u8_to_disp((w >> 16) & 0xff, scale), u8_to_disp(w >> 24, scale));
}
template <typename InT>
__device__ __forceinline__ float load1(const uint8_t *row, int col, float scale);
template <>
__device__ __forceinline__ float load1<float>(const uint8_t *row, int col, float) {
  return __ldcs(reinterpret_cast<const float *>(row) + col);
}
template <>
__device__ __forceinline__ float load1<uint8_t>(const uint8_t *row, int col, float scale) {
  return u8_to_disp(__ldcs(row + col), scale);
}

// Four pixels of one lane (columns u0, u0+32, u0+64, u0+96 of row v): the arithmetic is straight-line so the
// four FP64 dependency chains interleave; the rare slow path is one warp-level branch afterwards.
// xslow: bit k = column k of the lane must take the exact function, bit 4 + k = its numerator is +-0 (exact
// function only where the disparity is zero as well); yslow: bit 0 / bit 1, the same for the row.
template <int kMath>
__device__ __forceinline__ void points_of4(const QParams &Q, const double (&xd)[4], double yd, uint32_t xslow,
                                           uint32_t yslow, int u0, int v, const float (&d)[4], float4 (&p)[4]) {
  if constexpr (D2PC_IS_RECT(kMath)) {
    bool slow[4];
    const bool ys = (yslow & 1u) != 0u, yz = (yslow & 2u) != 0u;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if constexpr (kMath == kMathRect0Z)
        p[k] = reproject_exact_rectified<true, true, true>(Q, xd[k], yd, ys || ((xslow >> k) & 1u),
                                                           yz || ((xslow >> (4 + k)) & 1u), d[k], slow[k]);
      else
        p[k] = reproject_exact_rectified<kMath != kMathRectW, kMath == kMathRect0>(Q, xd[k], yd,
                                                                                   ys || ((xslow >> k) & 1u), false,
                                                                                   d[k], slow[k]);
    }
    if (__builtin_expect(slow[0] || slow[1] || slow[2] || slow[3], 0)) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (slow[k]) p[k] = reproject_exact_slow(Q.q, u0 + 32 * k, v, d[k]);
    }
  } else if constexpr (kMath == kMathGeneric) {
    bool slow[4];
    const double dv = (double)v;
#pragma unroll
    for (int k = 0; k < 4; ++k) p[k] = reproject_exact_generic_guarded(Q.q, (double)(u0 + 32 * k), dv, d[k], slow[k]);
    if (__builtin_expect(slow[0] || slow[1] || slow[2] || slow[3], 0)) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (slow[k]) p[k] = reproject_exact_slow(Q.q, u0 + 32 * k, v, d[k]);
    }
  } else if constexpr (kMath == kMathProbe) {
#pragma unroll
    for (int k = 0; k < 4; ++k) p[k] = make_float4(d[k], d[k], d[k], 1.0f);
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) p[k] = reproject_fast(Q.qf, u0 + 32 * k, v, d[k]);
  }
}

// Compaction form of points_of4 for the rectified Q with q33 == +-0 (band kernel): only survivors are stored, so
// the d == +-0 -> +-inf selects of the CROP form (and their per-column inf constants) are not computed at all.
// Classes, from the disparity bits alone:
//   fast   d_sure <= |d| < min(d_hi, inf): straight-line guarded multiply, the point is finite      -> kept
//   rest   any other non-zero finite |d| (sliver below d_sure, or >= d_hi): exact slow path decides -> rare
//   zero / inf / NaN disparity: never finite                                                       -> dropped
// A lane that meets anything rare (a "rest" pixel, a quotient next to a float rounding boundary, a degenerate
// row / column numerator) redoes its four pixels with the exact generic function, which is right for every
// input; keep[] then equals, pixel by pixel, what the band kernel's counting step derived from the same bits.
// The logic is spelled with unsigned arithmetic and one accumulated flag so that it stays in five predicates.
__device__ __forceinline__ uint32_t midpoint_distance(double q) {  // <= 0x20 next to a float rounding boundary
  return ((uint32_t)__double2loint(q) & 0x1fffffffu) - 0x0ffffff0u;
}
__device__ __forceinline__ void points_of4_keep(const QParams &Q, const double (&xd)[4], double yd, bool numer_slow,
                                                int u0, int v, const float (&d)[4], uint32_t sure_lo,
                                                uint32_t fast_span, float4 (&p)[4], bool (&keep)[4]) {
  bool rare = numer_slow;
  uint32_t cls[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint32_t mag = __float_as_uint(d[k]) & 0x7fffffffu;
    cls[k] = mag - sure_lo;  // fast class: cls < fast_span
    rare |= (cls[k] >= fast_span) && ((mag - 1u) < 0x7f7fffffu);
    const double w = __fma_rn(Q.q32, (double)d[k], 0.0);
    const double r = rcp_1ulp_inrange(w);  // garbage (never a trap) outside the fast class
    const double qx = __dmul_rn(xd[k], r), qy = __dmul_rn(yd, r), qz = __dmul_rn(Q.zd, r);
    // (a garbage quotient that happens to look ambiguous only sends the lane to the exact path)
    rare |= min(midpoint_distance(qx), min(midpoint_distance(qy), midpoint_distance(qz))) <= 0x20u;
    p[k].x = __double2float_rn(qx);
    p[k].y = __double2float_rn(qy);
    p[k].z = __double2float_rn(qz);
    p[k].w = 1.0f;  // pcl::PointXYZ's 4th float (cpp:74)
  }
  if (__builtin_expect(rare, 0)) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      p[k] = reproject_exact_slow(Q.q, u0 + 32 * k, v, d[k]);
      keep[k] = (cls[k] < fast_span) || point_is_finite(p[k]);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) keep[k] = cls[k] < fast_span;
  }
}

template <int kMath>
__device__ __forceinline__ float4 point_of(const QParams &Q, int u, int v, float d) {
  if constexpr (D2PC_IS_RECT(kMath)) {
    const double xd = rect_axis_const(u, Q.q03), yd = rect_axis_const(v, Q.q13);
    bool slow;
    float4 p = reproject_exact_rectified<kMath != kMathRectW, D2PC_IS_GUARD(kMath), kMath == kMathRect0Z>(
        Q, xd, yd, rect_axis_slow_t<kMath == kMathRect0Z>(xd) || rect_axis_slow_t<kMath == kMathRect0Z>(yd) || Q.zd_slow,
        rect_axis_zero(xd) || rect_axis_zero(yd), d, slow);
    if (__builtin_expect(slow, 0)) p = reproject_exact_slow(Q.q, u, v, d);
    return p;
  } else if constexpr (kMath == kMathGeneric) {
    return reproject_exact_generic(Q.q, u, v, d);
  } else {
    return reproject_fast(Q.qf, u, v, d);
  }
}

// ---------------------------------------------------------------------------
// CROP kernels
// ---------------------------------------------------------------------------
// What both CROP kernels (LDG rows below, TMA boxes further down) hold per work unit: column constants live in
// registers for the whole unit; row constants are computed by one lane per row and broadcast by shuffle.
template <int kMath>
struct CropCols {
  double xd[4];
  uint32_t xslow;
  double yd_lane;  // row constant of crop row r_base + lane
  double gcx[kMath == kMathGeneric ? 4 : 1][4];  // generic exact path: q[4i] * u of each of the lane's columns
};

template <int kMath>
__device__ __forceinline__ void crop_cols_init(CropCols<kMath> &c, const ReprojArgs &a, int c_base, int r_base,
                                               int lane) {
  const QParams &Q = a.Q;
  c.xslow = 0;
  c.yd_lane = 0.0;
  if constexpr (D2PC_IS_RECT(kMath)) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      c.xd[k] = rect_axis_const(a.border + c_base + 32 * k + lane, Q.q03);
      c.xslow |= rect_axis_slow_t<kMath == kMathRect0Z>(c.xd[k]) ? (1u << k) : 0u;
      if constexpr (kMath == kMathRect0Z) c.xslow |= rect_axis_zero(c.xd[k]) ? (16u << k) : 0u;
    }
    if (Q.zd_slow) c.xslow = 0xfu;
    c.yd_lane = rect_axis_const(a.border + r_base + lane, Q.q13);
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) c.xd[k] = 0.0;
  }
  if constexpr (kMath == kMathGeneric) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double du = (double)(a.border + c_base + 32 * k + lane);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        c.gcx[k][i] = __dmul_rn(Q.q[4 * i], du);
        asm volatile("" : "+d"(c.gcx[k][i]));  // keep the products in registers: ptxas would recompute them per pixel
      }
    }
  }
}

// The four points of crop row r_base + r of the unit, lane L owning columns L, L+32, L+64, L+96.
template <int kMath>
__device__ __forceinline__ void crop_row_points(const ReprojArgs &a, const CropCols<kMath> &c, int c_base, int r_base,
                                                int r, int lane, const float (&d)[4], float4 (&p)[4]) {
  const QParams &Q = a.Q;
  double yd = 0.0;
  uint32_t yslow = 0;
  if constexpr (D2PC_IS_RECT(kMath)) {
    yd = __shfl_sync(0xffffffffu, c.yd_lane, r);
    yslow = rect_axis_slow_t<kMath == kMathRect0Z>(yd) ? 1u : 0u;
    if constexpr (kMath == kMathRect0Z) yslow |= rect_axis_zero(yd) ? 2u : 0u;
  }
  if constexpr (kMath == kMathGeneric) {
    const int v = a.border + r_base + r, u0 = a.border + c_base + lane;
    const double dv = (double)v;
    double gry[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) gry[i] = __dmul_rn(Q.q[4 * i + 1], dv);
    bool slow[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) p[k] = reproject_exact_generic_hoisted(Q.q, c.gcx[k], gry, d[k], slow[k]);
    if (__builtin_expect(slow[0] || slow[1] || slow[2] || slow[3], 0)) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (slow[k]) p[k] = reproject_exact_slow(Q.q, u0 + 32 * k, v, d[k]);
    }
  } else {
    points_of4<kMath>(Q, c.xd, yd, c.xslow, yslow, a.border + c_base + lane, a.border + r_base + r, d, p);
  }
}

// Unit -> (frame, row block, segment) of the CROP kernels.
__device__ __forceinline__ void crop_unit(const ReprojArgs &a, uint32_t unit, uint32_t &f, int &rb, int &seg) {
  f = fastdiv(unit, a.div_upf);
  const uint32_t rem = unit - f * a.units_per_frame;
  rb = (int)fastdiv(rem, a.div_nseg);
  seg = (int)rem - rb * a.n_seg;
}

template <typename InT, bool kVec, int kMath, int kMinBlocks>
__global__ void __launch_bounds__(kThreads, kMinBlocks) reproject_crop_kernel(const __grid_constant__ ReprojArgs a) {
  __shared__ __align__(16) float stage[kWarpsPerCta][2][kSegCols];
  const int lane = threadIdx.x & 31;
  const int wic = threadIdx.x >> 5;

  // one work unit (128 crop columns x rows_per_unit crop rows) per warp; the hardware CTA scheduler balances
  const uint32_t unit = blockIdx.x * kWarpsPerCta + wic;
  if (unit >= a.total_units) return;
  uint32_t f;
  int rb, seg;
  crop_unit(a, unit, f, rb, seg);
  const int c_base = seg * kSegCols;
  const int r_base = rb * a.rows_per_unit;
  const int rows = min(a.rows_per_unit, a.ch - r_base);

  if constexpr (kVec && sizeof(InT) == 4) {
    // L2 prefetch of the unit a warp launched a fraction of a wave later will read (one 512-byte row per lane)
    if (a.prefetch_dist > 0 && lane < a.rows_per_unit) {
      const uint32_t u2 = unit + (uint32_t)a.prefetch_dist;  // total_units < 2^31 and the distance is clamped: no wrap
      if (u2 < a.total_units) {
        uint32_t f2;
        int rb2, seg2;
        crop_unit(a, u2, f2, rb2, seg2);
        const int row2 = rb2 * a.rows_per_unit + lane;
        const int cols2 = min(kSegCols, ((a.cw - seg2 * kSegCols) + 3) & ~3);
        if (row2 < a.ch)
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.in + (size_t)f2 * a.frame_stride +
                                                                        (size_t)(a.border + row2) * a.step +
                                                                        (size_t)(a.border + seg2 * kSegCols) * 4),
                       "r"((uint32_t)cols2 * 4u)
                       : "memory");
      }
    }
  }

  CropCols<kMath> cols;
  crop_cols_init(cols, a, c_base, r_base, lane);

  const uint8_t *in_row = a.in + (size_t)f * a.frame_stride + (size_t)(a.border + r_base) * a.step;
  float4 *out_row = a.out + (size_t)f * a.out_frame_stride + (size_t)r_base * a.cw;

  for (int r = 0; r < rows; r += 2, in_row += 2 * a.step, out_row += 2 * (size_t)a.cw) {
    // ---- load two crop rows of this segment
    float dd[2][4];
    if constexpr (kVec) {
      const int c4 = c_base + 4 * lane;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        if (r + j < rows && c4 < a.cw) {
          const float4 v = load4<InT>(in_row + (size_t)j * a.step, a.border + c4, a.scale);
          *reinterpret_cast<float4 *>(&stage[wic][j][4 * lane]) = v;
        }
      }
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int k = 0; k < 4; ++k) dd[j][k] = stage[wic][j][32 * k + lane];
      __syncwarp();
    } else {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int c = c_base + 32 * k + lane;
          dd[j][k] = (r + j < rows && c < a.cw) ? load1<InT>(in_row + (size_t)j * a.step, a.border + c, a.scale) : 1.0f;
        }
      }
    }
    // ---- compute + store: lane L owns columns L, L+32, L+64, L+96 -> each store is a 512-byte burst
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      if (r + j >= rows) break;
      float4 p[4];
      crop_row_points<kMath>(a, cols, c_base, r_base, r + j, lane, dd[j], p);
      float4 *o = out_row + (size_t)j * a.cw + c_base + lane;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (c_base + 32 * k + lane < a.cw) st_stream_f4(o + 32 * k, p[k]);
    }
  }
}

// ---------------------------------------------------------------------------
// CROP_FINITE kernel: order-preserving stream compaction, decoupled look-back
// ---------------------------------------------------------------------------
// A work unit is one crop row x 128 columns (one warp, 4 pixels per lane, same load + transpose as the CROP
// kernel).  Units are numbered in row-major order, so consecutive units are a contiguous range of the frame's
// point order.  A tile is kCIter x kCWarps = 32 consecutive units (<= 4096 pixels), one CTA per tile:
//   warp   reprojects its 4 units (all loads issued up front), parks the points in its own shared-memory cells
//          (SoA, conflict-free) and counts survivors with one __ballot_sync + popc per pixel slot;
//   block  32 unit counts -> warp-shuffle scan -> unit offsets and the tile total (one barrier);
//   grid   the tile total is published and the whole CTA runs the decoupled look-back (256 predecessors per
//          step) over 64-bit {epoch, flag, value} descriptors to get the tile's exclusive prefix;
//   warp   re-ballots its cells and stores survivors straight to their final place: every pixel slot is one
//          contiguous run of 16-byte points.
// Tiles never span frames; the look-back chain restarts at each frame.  Tile ids come from an atomic ticket, so
// every predecessor of a tile has already started (forward progress does not depend on CTA dispatch order).
// Descriptor: [63:34] launch epoch, [33:32] flag, [31:0] value.
constexpr int kCWarps = 8;
constexpr int kCThreads = kCWarps * 32;
constexpr int kCIter = 4;
constexpr int kTileUnits = kCWarps * kCIter;      // 32
constexpr int kTilePts = kTileUnits * kSegCols;   // 4096
constexpr size_t kCompactSmem = (size_t)kTilePts * 12 + (size_t)kCWarps * kSegCols * 4;  // 52 KB
constexpr uint32_t kFlagAggregate = 1, kFlagPrefix = 2;

__device__ __forceinline__ unsigned long long desc_pack(uint32_t epoch, uint32_t flag, uint32_t value) {
  return ((unsigned long long)epoch << 34) | ((unsigned long long)flag << 32) | value;
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long *p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// (double)(float)(i + q) for every image column / row, computed once per launch.  Entries the straight-line path
// must not use (tiny, inf, NaN numerators, and +-0 unless zero_ok: rect_axis_slow / rect_axis_slow_nz) are stored as
// NaN so consumers test one exponent field; the slow path recomputes from Q and never reads the table.  xtab is
// padded by kSegCols entries.
__global__ void rect_tables_kernel(double q03, double q13, int width, int height, bool zero_ok, double *xtab,
                                   double *ytab) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const double qnan = __longlong_as_double(0x7ff8000000000000ll);
  if (i < width + kSegCols) {
    const double x = rect_axis_const(i, q03);
    xtab[i] = (zero_ok ? rect_axis_slow_nz(x) : rect_axis_slow(x)) ? qnan : x;
  }
  if (i < height) {
    const double y = rect_axis_const(i, q13);
    ytab[i] = (zero_ok ? rect_axis_slow_nz(y) : rect_axis_slow(y)) ? qnan : y;
  }
}

template <typename InT, bool kVec, int kMath>
__global__ void __launch_bounds__(kCThreads, 4) reproject_compact_kernel(const __grid_constant__ ReprojArgs a) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  float *sx = reinterpret_cast<float *>(smem_raw);
  float *sy = sx + kTilePts;
  float *sz = sy + kTilePts;
  float *stage = sz + kTilePts;  // [kCWarps][128]
  __shared__ uint32_t unit_cnt[kTileUnits];
  __shared__ uint32_t lb_sum[kCWarps], lb_hit[kCWarps];
  __shared__ uint32_t s_tile;
  const int lane = threadIdx.x & 31, wic = threadIdx.x >> 5;
  const uint32_t lt_mask = (1u << lane) - 1u;
  const QParams &Q = a.Q;

  if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint32_t f = tile / a.tiles_per_frame;
  const uint32_t t_in_f = tile - f * a.tiles_per_frame;
  const uint8_t *in_f = a.in + (size_t)f * a.frame_stride;

  // ---- issue every load of this warp's kCIter units first
  int crow[kCIter], c_base[kCIter];
  bool unit_ok[kCIter];
  float4 raw[kCIter];
  float dds[kVec ? 1 : kCIter][4];
#pragma unroll
  for (int m = 0; m < kCIter; ++m) {
    const uint32_t unit = t_in_f * kTileUnits + m * kCWarps + wic;  // row-major (row, segment) index in the frame
    unit_ok[m] = unit < a.units_per_frame;
    crow[m] = unit_ok[m] ? (int)(unit / (uint32_t)a.n_seg) : 0;
    c_base[m] = unit_ok[m] ? (int)(unit - (uint32_t)crow[m] * a.n_seg) * kSegCols : 0;
    const uint8_t *in_row = in_f + (size_t)(a.border + crow[m]) * a.step;
    if constexpr (kVec) {
      const int c4 = c_base[m] + 4 * lane;
      raw[m] = (unit_ok[m] && c4 < a.cw) ? load4<InT>(in_row, a.border + c4, a.scale) : make_float4(1.f, 1.f, 1.f, 1.f);
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int c = c_base[m] + 32 * k + lane;
        dds[m][k] = (unit_ok[m] && c < a.cw) ? load1<InT>(in_row, a.border + c, a.scale) : 1.0f;
      }
    }
  }
  // ---- reproject, park, count
#pragma unroll
  for (int m = 0; m < kCIter; ++m) {
    float dd[4];
    if constexpr (kVec) {
      *reinterpret_cast<float4 *>(&stage[wic * kSegCols + 4 * lane]) = raw[m];
      __syncwarp();
#pragma unroll
      for (int k = 0; k < 4; ++k) dd[k] = stage[wic * kSegCols + 32 * k + lane];
      __syncwarp();
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) dd[k] = dds[m][k];
    }
    const int v = a.border + crow[m], u0 = a.border + c_base[m] + lane;
    double xd[4] = {0.0, 0.0, 0.0, 0.0}, yd = 0.0;
    uint32_t xslow = 0, yslow = 0;
    if constexpr (D2PC_IS_RECT(kMath)) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        xd[k] = a.xtab[u0 + 32 * k];  // padded table; NaN marks numerators for the slow path
        xslow |= (((uint32_t)__double2hiint(xd[k]) & 0x7ff00000u) == 0x7ff00000u) ? (1u << k) : 0u;
        if constexpr (kMath == kMathRect0Z) xslow |= rect_axis_zero(xd[k]) ? (16u << k) : 0u;
      }
      if (Q.zd_slow) xslow = 0xfu;
      yd = a.ytab[v];
      yslow = (((uint32_t)__double2hiint(yd) & 0x7ff00000u) == 0x7ff00000u) ? 1u : 0u;
      if constexpr (kMath == kMathRect0Z) yslow |= rect_axis_zero(yd) ? 2u : 0u;
    }
    float4 p[4];
    points_of4<kMath>(Q, xd, yd, xslow, yslow, u0, v, dd, p);
    uint32_t cnt = 0;
    const int cell0 = (m * kCWarps + wic) * kSegCols + lane;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const bool keep = unit_ok[m] && (c_base[m] + 32 * k + lane < a.cw) && point_is_finite(p[k]);
      cnt += __popc(__ballot_sync(0xffffffffu, keep));
      sx[cell0 + 32 * k] = keep ? p[k].x : __uint_as_float(0x7fc00000u);  // NaN marks a dropped cell
      sy[cell0 + 32 * k] = p[k].y;
      sz[cell0 + 32 * k] = p[k].z;
    }
    if (lane == 0) unit_cnt[m * kCWarps + wic] = cnt;
  }
  __syncthreads();
  // ---- 32 unit counts -> exclusive offsets (every warp scans; it is five shuffles)
  const uint32_t mine = lane < kTileUnits ? unit_cnt[lane] : 0u;
  uint32_t incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  const uint32_t tile_total = __shfl_sync(0xffffffffu, incl, 31);
  const uint32_t excl_unit = incl - mine;

  // ---- decoupled look-back, block-wide: 256 predecessors per step (thread j looks at tile t-1-j), so a chain
  // through every concurrently running tile resolves in two or three steps.  The first tile of a frame starts
  // the chain; predecessors before the frame start count as a zero prefix.
  unsigned long long *desc = a.tile_desc + tile;
  uint32_t excl = 0;
  if (t_in_f == 0) {
    if (threadIdx.x == 0) st_relaxed_u64(desc, desc_pack(a.epoch, kFlagPrefix, tile_total));
  } else {
    if (threadIdx.x == 0) st_relaxed_u64(desc, desc_pack(a.epoch, kFlagAggregate, tile_total));
    int look = (int)t_in_f - 1;
    for (;;) {
      const int my = look - (int)threadIdx.x;
      uint32_t flag = kFlagPrefix, val = 0;
      if (my >= 0) {
        unsigned long long dv;
        do {
          dv = ld_relaxed_u64(a.tile_desc + (tile - t_in_f) + my);
        } while ((uint32_t)(dv >> 34) != a.epoch || ((dv >> 32) & 3u) == 0);
        flag = (uint32_t)(dv >> 32) & 3u;
        val = (uint32_t)dv;
      }
      const uint32_t pmask = __ballot_sync(0xffffffffu, flag == kFlagPrefix);
      const int stop = pmask ? (__ffs(pmask) - 1) : 32;  // nearest predecessor in this warp's window with a prefix
      uint32_t contrib = (lane <= stop) ? val : 0u;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
      if (lane == 0) lb_sum[wic] = contrib, lb_hit[wic] = pmask ? 1u : 0u;
      __syncthreads();
      bool done = false;
#pragma unroll
      for (int w = 0; w < kCWarps; ++w) {
        if (!done) {
          excl += lb_sum[w];
          done = lb_hit[w] != 0u;
        }
      }
      if (done) break;
      look -= kCThreads;
      __syncthreads();  // lb_* are rewritten next step
    }
    if (threadIdx.x == 0) st_relaxed_u64(desc, desc_pack(a.epoch, kFlagPrefix, excl + tile_total));
  }
  if (threadIdx.x == 0 && t_in_f == a.tiles_per_frame - 1 && a.counts) a.counts[f] = excl + tile_total;
  // ---- survivors go straight to their final place; each pixel slot is one contiguous run
  float4 *out_f = a.out + (size_t)f * a.out_frame_stride + excl;
#pragma unroll
  for (int m = 0; m < kCIter; ++m) {
    uint32_t pos = __shfl_sync(0xffffffffu, excl_unit, m * kCWarps + wic);
    const int cell0 = (m * kCWarps + wic) * kSegCols + lane;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float x = sx[cell0 + 32 * k];
      const bool keep = (x == x);
      const uint32_t bal = __ballot_sync(0xffffffffu, keep);
      if (keep) st_stream_f4(out_f + pos + __popc(bal & lt_mask), make_float4(x, sy[cell0 + 32 * k], sz[cell0 + 32 * k], 1.0f));
      pos += __popc(bal);
    }
  }
}

// ---------------------------------------------------------------------------
// CROP_FINITE, rectified Q with q33 == +-0: band kernel (the default for this Q)
// ---------------------------------------------------------------------------
// One CTA owns a band of R full crop rows (a contiguous range of the frame's point order):
//   1. the band's disparities are brought into shared memory once with 16-byte cp.async (zero-filled past the
//      crop edge, so padding classifies as "dropped" without any mask);
//   2. every (row, 128-column) unit is classified from the disparity alone and counted -- no FP64 work yet.  For
//      this Q whether a point is finite is decided by the disparity for all but a sliver of inputs:
//        d == +-0, inf, NaN            -> W is +0 / NaN: the point is never finite              (dropped)
//        |d| >= d_sure (normal float)  -> |n / (q32*d)| < 2^127 for every numerator in the frame (kept); d_sure is
//                                         computed on the host from max |numerator| and |q32|
//        anything else (denormal, or |d| < d_sure ~ 2^-117)  -> decided by the exact slow path  (rare);
//   3. block scan of the unit counts -> unit offsets and the band total;
//   4. ONE decoupled look-back per band (block-wide, 256 predecessors per step);
//   5. warps sweep (segment, row-group) items: column numerators live in registers across the rows of the item,
//      points are reprojected from shared memory and the survivors stored straight to their final place.
// HBM traffic is exactly the algorithmic 4 B read + 16 B written per surviving point.
constexpr int kBandMaxUnits = 512;
constexpr int kBandMaxRows = 16;

// ---- mbarrier / TMA bulk-copy helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool mbar_test_wait(unsigned long long *bar, uint32_t parity) {  // non-blocking probe
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// Waiting consumers must not compete with the producer warps for issue slots: sleep between probes.
__device__ __forceinline__ void mbar_wait_backoff(unsigned long long *bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  do {
    __nanosleep(200);
  } while (!mbar_try_wait(bar, parity));
}
// TMA bulk copy global -> shared (1-D, 16-byte aligned, size a multiple of 16), completion counted on an mbarrier
__device__ __forceinline__ void tma_load_1d(uint32_t smem_dst, const void *gsrc, uint32_t bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void cp_async_16_zfill(void *smem_dst, const void *gmem_src, uint32_t src_bytes) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gmem_src), "r"(src_bytes) : "memory");
}

// kW warps per CTA (8 is what ships: four 46 KB CTAs per SM).  kZN: zero numerators stay straight-line (kMathRect0Z);
// a zero disparity is dropped here whatever its numerators, so no 0 / 0 case exists.
template <typename InT, bool kVec, int kMinB, int kW, bool kZN = false>
__global__ void __launch_bounds__(kW * 32, kMinB) reproject_compact_band_kernel(const __grid_constant__ ReprojArgs a) {
  constexpr int kT = kW * 32;
  extern __shared__ __align__(16) float sd[];  // [band_rows][cw_pad]
  __shared__ uint32_t unit_off[kBandMaxUnits];
  __shared__ double syd[kBandMaxRows];
  __shared__ uint32_t warp_tot[kW];
  __shared__ uint32_t lb_sum[kW], lb_hit[kW];
  __shared__ uint32_t s_tile;
  const int lane = threadIdx.x & 31, wic = threadIdx.x >> 5;
  const uint32_t lt_mask = (1u << lane) - 1u;
  const QParams &Q = a.Q;
  const int R = a.band_rows, cwp = a.cw_pad, n_seg = a.n_seg;

  constexpr bool kTma = kVec && sizeof(InT) == 4;  // aligned float rows: one TMA bulk copy per row
  __shared__ __align__(8) unsigned long long bar_rows;
  if (threadIdx.x == 0) {
    s_tile = atomicAdd(a.ticket, 1u);
    if constexpr (kTma) {
      mbar_init(&bar_rows, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint32_t f = tile / a.tiles_per_frame;
  const uint32_t t_in_f = tile - f * a.tiles_per_frame;
  const int row0 = (int)t_in_f * R;  // first crop row of the band
  const uint8_t *in_f = a.in + (size_t)f * a.frame_stride;

  // ---- 1. band -> shared memory
  const int rows_here = min(R, a.ch - row0);
  if constexpr (kTma) {
    // one cp.async.bulk per row, issued by a single thread, completion counted on an mbarrier; meanwhile all
    // threads zero what the copies do not write (padding columns up to cw_pad, rows past the frame's last crop
    // row), so that it classifies as "dropped" without any mask
    const int cw4 = (a.cw + 3) & ~3;
    if (threadIdx.x == 0) {
      mbar_arrive_expect_tx(&bar_rows, (uint32_t)rows_here * (uint32_t)cw4 * 4u);
      const uint8_t *src = in_f + (size_t)(a.border + row0) * a.step + (size_t)a.border * 4;
      for (int r = 0; r < rows_here; ++r)
        tma_load_1d(smem_u32(&sd[r * cwp]), src + (size_t)r * a.step, (uint32_t)cw4 * 4u, &bar_rows);
    }
    if (threadIdx.x == 32 && a.prefetch_dist > 0) {
      // pull the band that a CTA launched ~one wave later will need into L2, off everybody's critical path
      const uint64_t t2 = (uint64_t)tile + (uint64_t)a.prefetch_dist;
      if (t2 < (uint64_t)a.tiles_per_frame * (uint64_t)a.n_frames) {
        const uint32_t f2 = (uint32_t)(t2 / a.tiles_per_frame);
        const int row2 = (int)((uint32_t)t2 - f2 * a.tiles_per_frame) * R, rows2 = min(R, a.ch - row2);
        const uint8_t *src2 = a.in + (size_t)f2 * a.frame_stride + (size_t)(a.border + row2) * a.step + (size_t)a.border * 4;
        for (int r = 0; r < rows2; ++r)
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src2 + (size_t)r * a.step), "r"((uint32_t)cw4 * 4u)
                       : "memory");
      }
    }
    const int pad4 = (cwp - cw4) >> 2;  // float4 groups of padding per row
    for (int t = (int)threadIdx.x; t < pad4 * rows_here; t += kT) {
      const int r = t / pad4, g4 = t - r * pad4;
      *reinterpret_cast<float4 *>(&sd[r * cwp + cw4 + 4 * g4]) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int t = (int)threadIdx.x; t < (R - rows_here) * (cwp >> 2); t += kT)
      *reinterpret_cast<float4 *>(&sd[rows_here * cwp + 4 * t]) = make_float4(0.f, 0.f, 0.f, 0.f);
    mbar_wait(&bar_rows, 0);
    if (a.cw & 3)  // the copy brought up to 3 real pixels past the crop edge: they must not be counted or kept
      for (int t = (int)threadIdx.x; t < rows_here * 4; t += kT)
        if ((t & 3) >= (a.cw & 3)) sd[(t >> 2) * cwp + (a.cw & ~3) + (t & 3)] = 0.f;
  }
  // (cp.async / scalar staging for unaligned or mono8 rows: columns outer, rows inner)
  for (int c4 = 4 * (int)threadIdx.x; !kTma && c4 < cwp; c4 += 4 * kT) {
    const int left = min(max(a.cw - c4, 0), 4);  // crop pixels this 4-pixel group holds
    float *dst = &sd[c4];
    if constexpr (kVec && sizeof(InT) == 4) {
      const uint8_t *src = in_f + (size_t)(a.border + row0) * a.step + (size_t)(a.border + c4) * 4;
      if (left == 0) src = a.in;
      for (int r = 0; r < R; ++r, dst += cwp, src += a.step)
        cp_async_16_zfill(dst, r < rows_here ? (const void *)src : (const void *)a.in,
                          r < rows_here ? 4u * (uint32_t)left : 0u);
    } else {
      for (int r = 0; r < R; ++r, dst += cwp) {
        const uint8_t *in_row = in_f + (size_t)(a.border + row0 + r) * a.step;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < rows_here) {
          if (left > 0) v.x = load1<InT>(in_row, a.border + c4 + 0, a.scale);
          if (left > 1) v.y = load1<InT>(in_row, a.border + c4 + 1, a.scale);
          if (left > 2) v.z = load1<InT>(in_row, a.border + c4 + 2, a.scale);
          if (left > 3) v.w = load1<InT>(in_row, a.border + c4 + 3, a.scale);
        }
        *reinterpret_cast<float4 *>(dst) = v;
      }
    }
  }
  if ((int)threadIdx.x < R) {  // row numerators; NaN marks a row the straight-line path must not use
    const double y = rect_axis_const(a.border + row0 + (int)threadIdx.x, Q.q13);
    syd[threadIdx.x] = rect_axis_slow_t<kZN>(y) ? __longlong_as_double(0x7ff8000000000000ll) : y;
  }
  asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  // ---- 2. count the survivors of every unit (unit u = r * n_seg + s).  Only the total matters here, so a lane
  // takes four adjacent pixels (one 16-byte shared-memory load) and the warp sums with a single REDUX.
  const int n_units = R * n_seg;
  const uint32_t sure_lo = a.d_sure_bits, sure_span = 0x7f800000u - a.d_sure_bits;
  // straight-line class of step 5: d_sure <= |d| < min(d_hi, inf) (d_hi: see reproject_exact_rectified)
  const uint32_t fast_span = max(min(Q.dhi_bits, 0x7f800000u), sure_lo) - sure_lo;
  // The band is a flat array of units (cw_pad = n_seg * 128, so unit u starts at float 128 * u).  A warp takes
  // four consecutive units at a time; each lane counts its 4 pixels of every unit into one byte of a word and a
  // single REDUX adds all four units at once (a unit has 128 pixels, so no byte can carry into the next).
  for (int u0 = 4 * wic; u0 < n_units; u0 += 4 * kW) {
    uint32_t packed = 0;
    bool rare = false;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (u0 + q < n_units) {
        const float4 d4 = *reinterpret_cast<const float4 *>(&sd[(u0 + q) * kSegCols + 4 * lane]);
        const uint32_t m0 = __float_as_uint(d4.x) & 0x7fffffffu, m1 = __float_as_uint(d4.y) & 0x7fffffffu;
        const uint32_t m2 = __float_as_uint(d4.z) & 0x7fffffffu, m3 = __float_as_uint(d4.w) & 0x7fffffffu;
        // sure class: d_sure <= |d| < inf
        const uint32_t cq = ((m0 - sure_lo) < sure_span) + ((m1 - sure_lo) < sure_span) +
                            ((m2 - sure_lo) < sure_span) + ((m3 - sure_lo) < sure_span);
        rare |= min(min(m0 - 1u, m1 - 1u), min(m2 - 1u, m3 - 1u)) < sure_lo - 1u;  // sliver class 0 < |d| < d_sure
        packed |= cq << (8 * q);
      }
    }
    if (__builtin_expect(rare, 0)) {  // slivers are decided by the exact path
#pragma unroll 1
      for (int q = 0; q < 4 && u0 + q < n_units; ++q) {
        const int r = (u0 + q) / n_seg, sgm = (u0 + q) - r * n_seg;
        const float *px = &sd[(u0 + q) * kSegCols + 4 * lane];
#pragma unroll 1
        for (int e = 0; e < 4; ++e) {
          const uint32_t m = __float_as_uint(px[e]) & 0x7fffffffu;
          if ((m - 1u) < (sure_lo - 1u) &&
              point_is_finite(reproject_exact_slow(Q.q, a.border + sgm * kSegCols + 4 * lane + e, a.border + row0 + r, px[e])))
            packed += 1u << (8 * q);
        }
      }
    }
    packed = __reduce_add_sync(0xffffffffu, packed);
    if (lane < 4 && u0 + lane < n_units) unit_off[u0 + lane] = (packed >> (8 * lane)) & 0xffu;
  }
  __syncthreads();
  // ---- 3. exclusive scan of the unit counts (kE consecutive entries per thread)
  uint32_t band_total;
  {
    constexpr int kE = kBandMaxUnits / kT;
    const int i0 = kE * (int)threadIdx.x;
    uint32_t c[kE], sum = 0;
#pragma unroll
    for (int e = 0; e < kE; ++e) {
      c[e] = i0 + e < n_units ? unit_off[i0 + e] : 0u;
      sum += c[e];
    }
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    if (lane == 31) warp_tot[wic] = incl;
    __syncthreads();
    uint32_t wbase = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kW; ++w) {
      const uint32_t t = warp_tot[w];
      wbase += (w < wic) ? t : 0u;
      tot += t;
    }
    band_total = tot;
    uint32_t run = wbase + incl - sum;
#pragma unroll
    for (int e = 0; e < kE; ++e) {
      if (i0 + e < n_units) unit_off[i0 + e] = run;
      run += c[e];
    }
  }
  // ---- 4. decoupled look-back, block-wide; the first band of a frame starts the chain
  unsigned long long *desc = a.tile_desc + tile;
  uint32_t excl = 0;
  if (t_in_f == 0) {
    if (threadIdx.x == 0) st_relaxed_u64(desc, desc_pack(a.epoch, kFlagPrefix, band_total));
    __syncthreads();  // unit_off complete before step 5
  } else {
    if (threadIdx.x == 0) st_relaxed_u64(desc, desc_pack(a.epoch, kFlagAggregate, band_total));
    int look = (int)t_in_f - 1;
    for (;;) {
      const int my = look - (int)threadIdx.x;
      uint32_t flag = kFlagPrefix, val = 0;  // positions before the frame start act as a zero prefix
      if (my >= 0) {
        unsigned long long dv;
        do {
          dv = ld_relaxed_u64(a.tile_desc + (tile - t_in_f) + my);
        } while ((uint32_t)(dv >> 34) != a.epoch || ((dv >> 32) & 3u) == 0);
        flag = (uint32_t)(dv >> 32) & 3u;
        val = (uint32_t)dv;
      }
      const uint32_t pmask = __ballot_sync(0xffffffffu, flag == kFlagPrefix);
      const int stop = pmask ? (__ffs(pmask) - 1) : 32;
      uint32_t contrib = (lane <= stop) ? val : 0u;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
      if (lane == 0) lb_sum[wic] = contrib, lb_hit[wic] = pmask ? 1u : 0u;
      __syncthreads();
      bool done = false;
#pragma unroll
      for (int w = 0; w < kW; ++w) {
        if (!done) {
          excl += lb_sum[w];
          done = lb_hit[w] != 0u;
        }
      }
      if (done) break;
      look -= kT;
      __syncthreads();
    }
    if (threadIdx.x == 0) st_relaxed_u64(desc, desc_pack(a.epoch, kFlagPrefix, excl + band_total));
  }
  if (threadIdx.x == 0 && t_in_f == a.tiles_per_frame - 1 && a.counts) a.counts[f] = excl + band_total;

  // ---- 5. reproject + store: item = (segment, row group); column numerators stay in registers over its rows
  float4 *out_f = a.out + (size_t)f * a.out_frame_stride + excl;
  const int n_items = n_seg * a.band_groups;
  for (int item = wic; item < n_items; item += kW) {
    const int g = item / n_seg, sgm = item - g * n_seg;
    const int r_lo = g * a.group_rows, r_hi = min(r_lo + a.group_rows, R);
    const int u0 = a.border + sgm * kSegCols + lane;
    double xd[4];
    uint32_t xslow = Q.zd_slow ? 0xfu : 0u;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      xd[k] = rect_axis_const(u0 + 32 * k, Q.q03);
      xslow |= rect_axis_slow_t<kZN>(xd[k]) ? (1u << k) : 0u;
    }
    for (int r = r_lo; r < r_hi; ++r) {
      const double yd = syd[r];
      const bool yslow = ((uint32_t)__double2hiint(yd) & 0x7ff00000u) == 0x7ff00000u;
      const float *dp = &sd[r * cwp + sgm * kSegCols + lane];
      float dd[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) dd[k] = dp[32 * k];
      float4 p[4];
      bool kp[4];
      points_of4_keep(Q, xd, yd, yslow || xslow != 0u, u0, a.border + row0 + r, dd, sure_lo, fast_span, p, kp);
      uint32_t pos = unit_off[r * n_seg + sgm];
      if (__all_sync(0xffffffffu, kp[0] && kp[1] && kp[2] && kp[3])) {
        // the whole unit survives (the common case): four contiguous 512-byte bursts, no ranking (POPC shares the
        // quarter-rate XU pipe with the float64 conversions, which is this kernel's busiest pipe)
        float4 *o = out_f + pos + lane;
#pragma unroll
        for (int k = 0; k < 4; ++k) __stcs(o + 32 * k, p[k]);
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) pos = store_ranked_tight(out_f, pos, p[k], kp[k]);
      }
    }
  }
}


// ---------------------------------------------------------------------------
// CROP kernel, TMA form (aligned float rows, kR = 4 / 6 / 8 rows per unit)
// ---------------------------------------------------------------------------
// Same work units and 512-byte point stores as reproject_crop_kernel.  One lane per warp loads the unit's whole
// 128 x kR box into shared memory with one cp.async.bulk.tensor over a 3-D map (crop columns x crop rows x frames,
// encoded on the host, zero-filled past the crop edge) and issues one cp.async.bulk.prefetch.tensor.L2 for the
// unit prefetch_dist ahead.  Lanes then read their strided columns straight from the box: no per-row load,
// transpose or __syncwarp.  Full units (all but the last segment of a row and the last row block of a frame) run
// without row or column tests.
template <int kMath, int kMinBlocks, int kR>
__global__ void __launch_bounds__(kThreads, kMinBlocks) reproject_crop_tma_kernel(const __grid_constant__ ReprojArgs a) {
  __shared__ __align__(128) float box[kWarpsPerCta][kR * kSegCols];
  __shared__ __align__(8) unsigned long long bar[kWarpsPerCta];
  const int lane = threadIdx.x & 31;
  const int wic = threadIdx.x >> 5;
  const uint32_t unit = blockIdx.x * kWarpsPerCta + wic;
  if (unit >= a.total_units) return;
  uint32_t f;
  int rb, seg;
  crop_unit(a, unit, f, rb, seg);
  const int c_base = seg * kSegCols;
  const int r_base = rb * kR;
  const uint64_t tmap = reinterpret_cast<uint64_t>(&a.tmap);
  if (lane == 0) {
    mbar_init(&bar[wic], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_arrive_expect_tx(&bar[wic], kR * kSegCols * 4);  // out-of-bounds elements count too (zero-filled)
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], "
        "[%5];" ::"r"(smem_u32(box[wic])),
        "l"(tmap), "r"(c_base), "r"(r_base), "r"((int)f), "r"(smem_u32(&bar[wic]))
        : "memory");
    const uint32_t u2 = unit + (uint32_t)a.prefetch_dist;  // total_units < 2^31 and the distance is clamped: no wrap
    if (a.prefetch_dist > 0 && u2 < a.total_units) {
      uint32_t f2;
      int rb2, seg2;
      crop_unit(a, u2, f2, rb2, seg2);
      asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(tmap),
                   "r"(seg2 * kSegCols), "r"(rb2 * kR), "r"((int)f2)
                   : "memory");
    }
  }
  CropCols<kMath> cols;
  crop_cols_init(cols, a, c_base, r_base, lane);
  __syncwarp();  // the barrier is initialised before any lane waits on it
  mbar_wait(&bar[wic], 0);

  const float *bx = box[wic] + lane;
  // one 64-bit frame base, 32-bit offsets inside the frame (cw * ch < 2^31 where this kernel runs)
  float4 *o = a.out + (size_t)f * a.out_frame_stride + (uint32_t)(r_base * a.cw + c_base + lane);
  if (r_base + kR <= a.ch && c_base + kSegCols <= a.cw) {
#pragma unroll
    for (int r = 0; r < kR; ++r, o += a.cw) {
      float d[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) d[k] = bx[r * kSegCols + 32 * k];
      float4 p[4];
      crop_row_points<kMath>(a, cols, c_base, r_base, r, lane, d, p);
#pragma unroll
      for (int k = 0; k < 4; ++k) st_stream_f4(o + 32 * k, p[k]);
    }
  } else {
    const int rows = min(kR, a.ch - r_base);
#pragma unroll 1
    for (int r = 0; r < rows; ++r, o += a.cw) {
      float d[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) d[k] = bx[r * kSegCols + 32 * k];
      float4 p[4];
      crop_row_points<kMath>(a, cols, c_base, r_base, r, lane, d, p);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (c_base + 32 * k + lane < a.cw) st_stream_f4(o + 32 * k, p[k]);
    }
  }
}

template <int kMath, int kMinBlocks>
void launch_crop_tma(const ReprojArgs &a, int grid, cudaStream_t s) {
  switch (a.rows_per_unit) {
    case 4: reproject_crop_tma_kernel<kMath, kMinBlocks, 4><<<grid, kThreads, 0, s>>>(a); break;
    case 6: reproject_crop_tma_kernel<kMath, kMinBlocks, 6><<<grid, kThreads, 0, s>>>(a); break;
    default: reproject_crop_tma_kernel<kMath, kMinBlocks, 8><<<grid, kThreads, 0, s>>>(a); break;
  }
}

template <typename K>
cudaError_t launch_compact(K kernel, const ReprojArgs &a, int grid, cudaStream_t s) {
  // 52 KB of dynamic shared memory needs the opt-in on every instantiation (and on every device)
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCompactSmem);
  if (e != cudaSuccess) return e;
  kernel<<<grid, kCThreads, kCompactSmem, s>>>(a);
  return cudaGetLastError();
}

template <typename InT, int kMath>
cudaError_t launch_typed(const ReprojArgs &a, bool vec, bool compact, int grid, int min_blocks, cudaStream_t s) {
  if constexpr (sizeof(InT) == 4) {
    if (a.tma) {
      switch (min_blocks) {
        case 4: launch_crop_tma<kMath, 4>(a, grid, s); break;
        case 6: launch_crop_tma<kMath, 6>(a, grid, s); break;
        case 8: launch_crop_tma<kMath, 8>(a, grid, s); break;
        default: launch_crop_tma<kMath, 7>(a, grid, s); break;
      }
      return cudaGetLastError();
    }
  }
  if (compact) {
    if constexpr (kMath == kMathProbe) return cudaErrorInvalidValue;  // a CROP-kernel hook only
    if constexpr (D2PC_IS_GUARD(kMath)) {
      if (a.d_sure_bits != 0 && a.band_rows > 0) {  // band kernel
        constexpr bool kZN = kMath == kMathRect0Z;
        const size_t smem = (size_t)a.band_rows * a.cw_pad * sizeof(float);
        auto kern = !vec ? reproject_compact_band_kernel<InT, false, 3, 8, kZN>
                         : (min_blocks == 3 ? reproject_compact_band_kernel<InT, true, 3, 8, kZN>
                                            : reproject_compact_band_kernel<InT, true, 4, 8, kZN>);
        if (smem > 48 * 1024) {
          cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
          if (e != cudaSuccess) return e;
        }
        kern<<<grid, kCThreads, smem, s>>>(a);
        return cudaGetLastError();
      }
    }
    if constexpr (kMath != kMathProbe)
      return vec ? launch_compact(reproject_compact_kernel<InT, true, kMath>, a, grid, s)
                 : launch_compact(reproject_compact_kernel<InT, false, kMath>, a, grid, s);
  } else if (vec) {
    switch (min_blocks) {  // 128-thread CTAs: 4 -> <=128 regs, 6 -> 80, 7 -> 72, 8 -> 64
      case 4: reproject_crop_kernel<InT, true, kMath, 4><<<grid, kThreads, 0, s>>>(a); break;
      case 6: reproject_crop_kernel<InT, true, kMath, 6><<<grid, kThreads, 0, s>>>(a); break;
      case 8: reproject_crop_kernel<InT, true, kMath, 8><<<grid, kThreads, 0, s>>>(a); break;
      default: reproject_crop_kernel<InT, true, kMath, 7><<<grid, kThreads, 0, s>>>(a); break;
    }
  } else {
    reproject_crop_kernel<InT, false, kMath, 6><<<grid, kThreads, 0, s>>>(a);
  }
  return cudaGetLastError();
}

}  // namespace

// Host: classify Q (disparity_to_point_cloud.hpp:90-104 produces the rectified form).
void make_qparams(const double q[16], QParams *out) {
  QParams P{};
  for (int i = 0; i < 16; ++i) {
    P.q[i] = q[i];
    P.qf[i] = (float)q[i];
  }
  auto bits = [](double x) {
    uint64_t b;
    memcpy(&b, &x, 8);
    return b;
  };
  auto pzero = [&](double x) { return bits(x) == 0; };
  auto fin = [](double x) { return x == x && x - x == 0.0; };
  const double a32 = q[14] < 0 ? -q[14] : q[14];
  const bool rect = q[0] == 1.0 && pzero(q[1]) && pzero(q[2]) && pzero(q[4]) && q[5] == 1.0 && pzero(q[6]) &&
                    pzero(q[8]) && pzero(q[9]) && pzero(q[10]) && pzero(q[12]) && pzero(q[13]) && fin(q[3]) &&
                    fin(q[7]) && fin(q[11]) && fin(q[15]) && fin(q[14]) && a32 > 1e-30 && a32 < 1e30;
  P.rectified = rect ? 1 : 0;
  P.q03 = q[3];
  P.q13 = q[7];
  P.q32 = q[14];
  P.q33 = q[15];
  P.q33_zero = (q[15] == 0.0) ? 1 : 0;
  {
    float dhi = (float)(0x1p64 / (a32 > 0 ? a32 : 1.0));
    if (!(dhi < 3.0e38f)) dhi = 3.0e38f;
    if (dhi < 0x1p-125f) dhi = 0x1p-125f;
    memcpy(&P.dhi_bits, &dhi, 4);
  }
  // h2 = ((0*u + 0*v) + 0*d) + q23 = (+0) + q23 for finite u, v >= 0 and finite d
  volatile double z = 0.0;
  const double h2 = z + q[11];
  P.zd = (double)(float)h2;
  const uint64_t zb = bits(P.zd);
  P.zd_slow = (((zb >> 52) & 0x7ff) == 0x7ff || ((zb >> 52) & 0x7ff) < 1023 - 40) ? 1 : 0;  // as rect_axis_slow
  {
    uint32_t zi = (zb << 1) == 0 ? 0xFFC00000u : (uint32_t)(((zb >> 63) << 31) | 0x7f800000u);
    memcpy(&P.zinf, &zi, 4);
  }
  *out = P;
}

static uint64_t compact_tiles_per_frame(long cw, long ch) {
  const uint64_t n_seg = (uint64_t)((cw + kSegCols - 1) / kSegCols);
  return (n_seg * (uint64_t)ch + kTileUnits - 1) / kTileUnits;
}

// tile descriptors (must start zeroed: epoch 0 means "never written")
size_t reproject_scratch_bytes(uint32_t n_frames, uint32_t width, uint32_t height, int border) {
  const long cw = (long)width - 2L * border, ch = (long)height - 2L * border;
  // enough for either tiling: 32-unit tiles (park kernel) or row bands (band kernel)
  const uint64_t tiles = (cw > 0 && ch > 0) ? std::max<uint64_t>(compact_tiles_per_frame(cw, ch), (uint64_t)ch) : 0;
  return (size_t)(tiles * n_frames * 8 + 256);
}
// per-column / per-row numerator tables of the rectified path
size_t reproject_table_bytes(uint32_t width, uint32_t height) { return ((size_t)width + kSegCols + height) * 8 + 64; }

// Which arithmetic a launch takes (host side, from Q and the knobs).
static int select_math(const ReprojectLaunch &L) {
  const QParams &Q = *L.Q;
  // X is exactly zero on an image column (an integral principal point): keep that column straight-line
  auto zero_column = [&]() {
    const double c = std::nearbyint(-Q.q03);
    return c >= 0.0 && c < (double)L.width && (float)(c + Q.q03) == 0.0f;
  };
  const bool zero_numer = L.zero_numer > 0 || (L.zero_numer == 0 && zero_column());
  return L.arith_fast ? kMathFast
         : (Q.rectified && !L.force_generic
                ? (Q.q33_zero ? (L.exact_variant == 1 ? kMathRect0M : (zero_numer ? kMathRect0Z : kMathRect0)) : kMathRectW)
                : kMathGeneric);
}

bool reproject_fuses_with_median(const ReprojectLaunch &L, bool *zero_numer) {
  if (!L.Q || L.compact || L.Q->zd_slow) return false;
  const int math = select_math(L);
  if (zero_numer) *zero_numer = math == kMathRect0Z;
  return D2PC_IS_GUARD(math);
}

// 3-D tiled map of the crop region (columns x rows x frames, 4-byte elements) with a 128 x rows x 1 box.
// cuTensorMapEncodeTiled comes through the runtime's driver entry point, so the library links no libcuda.
static bool encode_crop_map(CUtensorMap *m, const ReprojectLaunch &L, long cw, long ch, int rows) {
  static const PFN_cuTensorMapEncodeTiled_v12000 encode = [] {
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    return cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &fn, 12000, cudaEnableDefault, &q) ==
                       cudaSuccess &&
                   q == cudaDriverEntryPointSuccess
               ? reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn)
               : nullptr;
  }();
  if (!encode) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)cw, (cuuint64_t)ch, (cuuint64_t)L.n_frames};
  // a lone frame's stride is never stepped over; any valid one will do
  const cuuint64_t strides[2] = {(cuuint64_t)L.step, L.n_frames > 1 ? (cuuint64_t)L.frame_stride : (cuuint64_t)L.step * ch};
  const cuuint32_t box[3] = {(cuuint32_t)kSegCols, (cuuint32_t)rows, 1u}, elem[3] = {1u, 1u, 1u};
  const uint8_t *base = static_cast<const uint8_t *>(L.in) + (size_t)L.border * L.step + (size_t)L.border * 4;
  return encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<uint8_t *>(base), dims, strides, box, elem,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

cudaError_t launch_reproject(const ReprojectLaunch &L, cudaStream_t stream, int *launches) {
  const long cw = (long)L.width - 2L * L.border, ch = (long)L.height - 2L * L.border;
  if (launches) *launches = 0;
  if (cw <= 0 || ch <= 0 || L.n_frames == 0) {
    // nothing kept: the reference publishes an empty cloud
    if (L.counts && L.n_frames) {
      if (launches) *launches = 0;
      return cudaMemsetAsync(L.counts, 0, sizeof(uint32_t) * L.n_frames, stream);
    }
    return cudaSuccess;
  }
  ReprojArgs a{};
  a.in = static_cast<const uint8_t *>(L.in);
  a.step = L.step;
  a.frame_stride = L.frame_stride;
  a.out = reinterpret_cast<float4 *>(L.out);
  a.out_frame_stride = L.out_stride_bytes / 16;
  a.counts = L.counts;
  a.n_frames = (int)L.n_frames;
  a.width = (int)L.width;
  a.height = (int)L.height;
  a.border = L.border;
  a.cw = (int)cw;
  a.ch = (int)ch;
  a.scale = L.scale;
  a.Q = *L.Q;

  const int esz = L.in_is_f32 ? 4 : 1;
  // 16-byte (float) / 4-byte (mono8) vector loads need aligned rows; a row tail may read up to 3 pixels past the
  // crop edge, which stays inside the frame row only if the border is at least 3 wide.
  const size_t valign = L.in_is_f32 ? 16 : 4;
  const bool vec = (reinterpret_cast<uintptr_t>(L.in) % valign == 0) && (L.step % valign == 0) &&
                   (L.frame_stride % valign == 0) && ((size_t)L.border * esz % valign == 0) &&
                   (cw % 4 == 0 || L.border >= 3) && !L.force_scalar;

  int math = select_math(L);
  const bool compact = L.compact;

  int grid;
  a.n_seg = (int)((cw + kSegCols - 1) / kSegCols);
  if (compact) {
    a.units_per_frame = (uint32_t)a.n_seg * (uint32_t)ch;
    a.tiles_per_frame = (uint32_t)compact_tiles_per_frame(cw, ch);
    a.tile_desc = static_cast<unsigned long long *>(L.scratch);
    double *tabs = static_cast<double *>(L.tables);
    a.xtab = tabs;
    a.ytab = tabs + L.width + kSegCols;
    a.ticket = L.ticket;
    a.epoch = L.epoch;
    const uint64_t total = (uint64_t)a.tiles_per_frame * L.n_frames;
    if (total > 0xffffffffull) return cudaErrorInvalidValue;
    grid = (int)total;  // one CTA per tile; the ticket, not blockIdx, names the tile
    cudaError_t e = cudaMemsetAsync(a.ticket, 0, sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    if (D2PC_IS_GUARD(math) && !a.Q.zd_slow && L.compact_variant != 1) {
      // |n| <= max_numer for every numerator of the frame; |q| = |n| / (|q32| * |d|) < 2^127 once
      // |d| >= max_numer * 2^-127 / |q32|; doubled for margin, clamped to the smallest normal float.
      const double aq32 = a.Q.q32 < 0 ? -a.Q.q32 : a.Q.q32;
      auto mag = [](double x) { return x < 0 ? -x : x; };
      double max_numer = mag(a.Q.zd);
      max_numer = std::max(max_numer, mag(a.Q.q03) + (double)L.width + 1.0);
      max_numer = std::max(max_numer, mag(a.Q.q13) + (double)L.height + 1.0);
      double d_sure = 2.0 * max_numer * 0x1p-127 / aq32;
      if (d_sure < 0x1p-126) d_sure = 0x1p-126;
      if (d_sure < 3.0e38) {
        float fs = (float)d_sure;
        if ((double)fs < d_sure) fs = std::nextafter(fs, INFINITY);
        memcpy(&a.d_sure_bits, &fs, 4);
      }
    }
    if (a.d_sure_bits != 0 && L.compact_variant != 1) {
      // band geometry: R rows per CTA (<= ~46 KB of disparities, <= 512 units), split into row groups so that
      // (segments x groups) fills the 8 warps evenly
      a.cw_pad = a.n_seg * kSegCols;
      const size_t row_bytes = (size_t)a.cw_pad * sizeof(float);
      // four 8-warp CTAs of <= 46 KB per SM.  (Measured in round 2: eight 4-warp CTAs of <= 24 KB are slower, 0.79 vs
      // 0.84 at 720p and 0.74 vs 0.90 at 4K, and so are smaller bands at 8 warps -- 4 rows: 0.65 -- the per-band
      // fixed cost (ticket, row loads, scan, look-back) wants bands as large as the shared memory of 4 CTAs allows.)
      const int bw = kCWarps;
      int r_max = (int)std::min<size_t>((46 * 1024) / row_bytes, (size_t)kBandMaxRows);
      r_max = std::min(r_max, kBandMaxUnits / a.n_seg);
      if (r_max < 1 && row_bytes <= 200 * 1024 && a.n_seg <= kBandMaxUnits) r_max = 1;
      if (r_max > (int)ch) r_max = (int)ch;
      if (L.rows_per_unit > 0 && L.rows_per_unit < r_max) r_max = L.rows_per_unit;  // tuning knob
      double best = -1.0;
      for (int r = r_max; r >= 1 && r >= r_max - 3; --r)
        for (int g = 1; g <= r; ++g) {
          const int gr = (r + g - 1) / g, ga = (r + gr - 1) / gr;
          const int items = a.n_seg * ga;
          const double eff = (double)items / (bw * ((items + bw - 1) / bw));
          const double score = eff * (gr / (gr + 0.6)) * (r / (r + 0.5));
          if (score > best + 1e-9) best = score, a.band_rows = r, a.band_groups = ga, a.group_rows = gr;
        }
      if (a.band_rows > 0) {
        a.tiles_per_frame = (uint32_t)((ch + a.band_rows - 1) / a.band_rows);
        const uint64_t total_b = (uint64_t)a.tiles_per_frame * L.n_frames;
        if (total_b > 0xffffffffull) return cudaErrorInvalidValue;
        grid = (int)total_b;
        a.prefetch_dist = L.prefetch_dist < 0 ? 0 : (L.prefetch_dist > 0 ? L.prefetch_dist : L.sm_count);  // measured plateau: 100-300 tiles
      }
    }
    if (a.Q.rectified && !L.arith_fast && !L.force_generic && a.band_rows == 0) {
      const int n = (int)(L.width + kSegCols > L.height ? L.width + kSegCols : L.height);
      rect_tables_kernel<<<(n + 255) / 256, 256, 0, stream>>>(a.Q.q03, a.Q.q13, (int)L.width, (int)L.height,
                                                            math == kMathRect0Z, tabs, tabs + L.width + kSegCols);
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
      if (launches) *launches += 1;
    }
  } else {
    // rows per unit: large units amortise the per-unit constants, small ones spread a lone frame over the chip.
    // TMA boxes make a unit's fixed cost small enough that 4-row units win under the sustained power cap as well
    // (4K x 16, 320 launches: 369 us against 375 at 8 rows; the per-row loads want 8: 381 against 390).
    const bool tma_rows = vec && L.in_is_f32 && L.crop_load == 0;
    int rb = L.rows_per_unit > 0 ? L.rows_per_unit : (tma_rows ? 4 : 8);
    const uint64_t want_units = (uint64_t)L.sm_count * 32;
    while (rb > 2 && (uint64_t)a.n_seg * ((ch + rb - 1) / rb) * L.n_frames < want_units) rb >>= 1;
    if (rb > 32) rb = 32;
    rb &= ~1;
    if (rb < 2) rb = 2;
    a.rows_per_unit = rb;
    a.n_rb = (int)((ch + rb - 1) / rb);
    a.units_per_frame = (uint32_t)a.n_seg * (uint32_t)a.n_rb;
    const uint64_t total = (uint64_t)a.units_per_frame * L.n_frames;
    if (total >= 0x7fffffffull) return cudaErrorInvalidValue;  // fastdiv's domain (8 M units are 1024 4K frames)
    a.total_units = (uint32_t)total;
    a.div_upf = make_fastdiv(a.units_per_frame);
    a.div_nseg = make_fastdiv((uint32_t)a.n_seg);
    grid = (int)((total + kWarpsPerCta - 1) / kWarpsPerCta);
    // L2 prefetch distance in units (~4100 units are in flight; measured plateau 256-2048)
    a.prefetch_dist = L.prefetch_dist < 0 ? 0 : (L.prefetch_dist > 0 ? std::min(L.prefetch_dist, 1 << 24) : 512);
    // TMA box loads where the map can describe the rows (the LDG kernel serves every other case)
    a.tma = tma_rows && (rb == 4 || rb == 6 || rb == 8) &&
            (uint64_t)cw * (uint64_t)ch < (1ull << 31) && encode_crop_map(&a.tmap, L, cw, ch, rb);
  }
  if (L.crop_probe && !compact) {
    if (!L.in_is_f32) return cudaErrorInvalidValue;
    math = kMathProbe;
  }
  // the generic exact path keeps 16 column products in registers: 4 CTAs per SM (<= 128 registers).  The others:
  // 6 CTAs (80 registers) beat 7 (72, more spills) by 0.5 % in every sustained and burst A/B of round 2
  // (profiles/r2_crop_rows_power.txt); 8 (64 registers) is 5 % slower.
  const int min_blocks = L.ctas_per_sm > 0 ? L.ctas_per_sm : (math == kMathGeneric && !compact ? 4 : 6);
  if (launches) *launches += 1;

#define D2PC_DISPATCH(T)                                                          \
  switch (math) {                                                                 \
    case kMathRect0: return launch_typed<T, kMathRect0>(a, vec, compact, grid, min_blocks, stream); \
    case kMathRect0Z: return launch_typed<T, kMathRect0Z>(a, vec, compact, grid, min_blocks, stream); \
    case kMathRect0M: return launch_typed<T, kMathRect0M>(a, vec, compact, grid, min_blocks, stream); \
    case kMathRectW: return launch_typed<T, kMathRectW>(a, vec, compact, grid, min_blocks, stream); \
    case kMathGeneric: return launch_typed<T, kMathGeneric>(a, vec, compact, grid, min_blocks, stream); \
    default: return launch_typed<T, kMathFast>(a, vec, compact, grid, min_blocks, stream);    \
  }
  if (L.in_is_f32) {
    if (math == kMathProbe) return launch_typed<float, kMathProbe>(a, vec, compact, grid, min_blocks, stream);
    D2PC_DISPATCH(float)
  } else {
    D2PC_DISPATCH(uint8_t)
  }
#undef D2PC_DISPATCH
}

}  // namespace d2pc
