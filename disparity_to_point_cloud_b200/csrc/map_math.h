/* map_math.h -- the key, centre, norm and ray (DDA) math of the occupancy map (include/d2pc_b200.h, "occupancy map"),
 * one source for the CUDA kernels (csrc/occupancy.cu) and the C reference (tests/map_ref/occupancy.c), so the two meet
 * key for key.
 *
 * Every operation is one IEEE-754 operation rounded to nearest on its own: explicit __f*_rn / __d*_rn on the device,
 * plain operators on the host, where the file must be compiled with -ffp-contract=off.  The float / double mix is
 * octomap's as restated in the header: float point3d arithmetic, double keys, centres and ray parameters.
 *
 *   d2pc_map_key(rf, c, &k)   k = (int)floor(rf * (double)c) + 32768, valid only when 0 <= k < 65536
 *                             (OcTreeBaseImpl::coordToKeyChecked, rf = 1.0 / resolution in double).
 *   d2pc_map_centre(k, res)   ((double)(k - 32768) + 0.5) * res (keyToCoord at full depth).
 *   d2pc_map_node_size / d2pc_map_node_centre   getNodeSize(depth) and keyToCoord(k, depth) of a coarser node.
 *   d2pc_map_norm(x, y, z)    sqrt((double)((x*x + y*y) + z*z)): float products and sums, no FMA, a double sqrt
 *                             (octomath Vector3::norm).
 *   d2pc_map_ray_begin/next   OcTreeBaseImpl::computeRayKeys step by step: begin yields the origin's key, each next
 *                             one more free cell, until the end key or min(tMax) > length.
 * One guard the reference does not have: a ray stops after kD2pcMapRayMaxSteps steps.  No ray between two valid keys
 * takes that many (each axis moves at most 65535 keys); the bound only matters for a direction that overflows float
 * (a resolution near 1e14 m), where computeRayKeys would loop forever. */
#ifndef D2PC_MAP_MATH_H_
#define D2PC_MAP_MATH_H_

#include <float.h>
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define D2PC_MM_FN static __host__ __device__ __forceinline__
#else
#define D2PC_MM_FN static inline
#endif

#if defined(__CUDA_ARCH__)
#define D2PC_MM_FADD(a, b) __fadd_rn((a), (b))
#define D2PC_MM_FSUB(a, b) __fsub_rn((a), (b))
#define D2PC_MM_FMUL(a, b) __fmul_rn((a), (b))
#define D2PC_MM_FDIV(a, b) __fdiv_rn((a), (b))
#define D2PC_MM_DADD(a, b) __dadd_rn((a), (b))
#define D2PC_MM_DSUB(a, b) __dsub_rn((a), (b))
#define D2PC_MM_DMUL(a, b) __dmul_rn((a), (b))
#define D2PC_MM_DDIV(a, b) __ddiv_rn((a), (b))
#define D2PC_MM_DSQRT(a) __dsqrt_rn(a)
#define D2PC_MM_D2F(a) __double2float_rn(a)
#else
#define D2PC_MM_FADD(a, b) ((a) + (b))
#define D2PC_MM_FSUB(a, b) ((a) - (b))
#define D2PC_MM_FMUL(a, b) ((a) * (b))
#define D2PC_MM_FDIV(a, b) ((a) / (b))
#define D2PC_MM_DADD(a, b) ((a) + (b))
#define D2PC_MM_DSUB(a, b) ((a) - (b))
#define D2PC_MM_DMUL(a, b) ((a) * (b))
#define D2PC_MM_DDIV(a, b) ((a) / (b))
#define D2PC_MM_DSQRT(a) sqrt(a)
#define D2PC_MM_D2F(a) ((float)(a))
#endif

#define kD2pcMapRayMaxSteps (3u * 65536u)

/* coordToKeyChecked on one axis: 1 and *k when the key is valid, else 0 */
D2PC_MM_FN int d2pc_map_key(double rf, float c, uint16_t *k) {
  const double v = floor(D2PC_MM_DMUL(rf, (double)c));
  if (!(v >= -32768.0 && v < 32768.0)) return 0; /* NaN fails too */
  *k = (uint16_t)((int)v + 32768);
  return 1;
}

D2PC_MM_FN int d2pc_map_key3(double rf, float x, float y, float z, uint16_t k[3]) {
  return d2pc_map_key(rf, x, &k[0]) && d2pc_map_key(rf, y, &k[1]) && d2pc_map_key(rf, z, &k[2]);
}

D2PC_MM_FN double d2pc_map_centre(uint16_t k, double res) {
  return D2PC_MM_DMUL(D2PC_MM_DADD((double)((int)k - 32768), 0.5), res);
}

/* OcTreeBaseImpl::getNodeSize(depth): res * (double)(1 << (16 - depth)), depth 0 (the root) .. 16 (a voxel) */
D2PC_MM_FN double d2pc_map_node_size(uint32_t depth, double res) {
  return D2PC_MM_DMUL(res, (double)(1u << (16u - depth)));
}

/* OcTreeBaseImpl::keyToCoord(k, depth): the centre of the depth-`depth` node that holds key k (any key inside the
 * node gives the same floor).  0 at the root, d2pc_map_centre at full depth. */
D2PC_MM_FN double d2pc_map_node_centre(uint16_t k, uint32_t depth, double res) {
  if (depth == 0) return 0.0;
  if (depth == 16) return d2pc_map_centre(k, res);
  const double q = floor(D2PC_MM_DDIV(D2PC_MM_DSUB((double)k, 32768.0), (double)(1u << (16u - depth))));
  return D2PC_MM_DMUL(D2PC_MM_DADD(q, 0.5), d2pc_map_node_size(depth, res));
}

D2PC_MM_FN double d2pc_map_norm(float x, float y, float z) {
  const float s = D2PC_MM_FADD(D2PC_MM_FADD(D2PC_MM_FMUL(x, x), D2PC_MM_FMUL(y, y)), D2PC_MM_FMUL(z, z));
  return D2PC_MM_DSQRT((double)s);
}

/* computeRayKeys' state: the current key, the end key and the DDA's per-axis step, tMax and tDelta */
typedef struct d2pc_map_ray {
  uint16_t key[3], end[3];
  int step[3];
  double tmax[3], tdelta[3];
  double length; /* (double)(float)norm(e - o) */
  uint32_t steps;
} d2pc_map_ray;

/* 0: the ray is empty (a key is invalid, or o and e share one).  1: r->key is the origin's key, the ray's first cell. */
D2PC_MM_FN int d2pc_map_ray_begin(d2pc_map_ray *r, const float o[3], const float e[3], double res, double rf) {
  if (!d2pc_map_key3(rf, o[0], o[1], o[2], r->key) || !d2pc_map_key3(rf, e[0], e[1], e[2], r->end)) return 0;
  if (r->key[0] == r->end[0] && r->key[1] == r->end[1] && r->key[2] == r->end[2]) return 0;
  float d[3] = {D2PC_MM_FSUB(e[0], o[0]), D2PC_MM_FSUB(e[1], o[1]), D2PC_MM_FSUB(e[2], o[2])};
  const float length = D2PC_MM_D2F(d2pc_map_norm(d[0], d[1], d[2]));
  for (int i = 0; i < 3; ++i) d[i] = D2PC_MM_FDIV(d[i], length);
  for (int i = 0; i < 3; ++i) {
    r->step[i] = d[i] > 0.0f ? 1 : d[i] < 0.0f ? -1 : 0;
    if (r->step[i] != 0) {
      const float half = D2PC_MM_D2F(D2PC_MM_DMUL(D2PC_MM_DMUL((double)r->step[i], res), 0.5));
      const double border = D2PC_MM_DADD(d2pc_map_centre(r->key[i], res), (double)half);
      r->tmax[i] = D2PC_MM_DDIV(D2PC_MM_DSUB(border, (double)o[i]), (double)d[i]);
      r->tdelta[i] = D2PC_MM_DDIV(res, (double)fabsf(d[i]));
    } else {
      r->tmax[i] = DBL_MAX;
      r->tdelta[i] = DBL_MAX;
    }
  }
  r->length = (double)length;
  r->steps = 0;
  return 1;
}

/* One DDA step: 1 when the new r->key is a free cell of the ray, 0 when the ray has ended. */
D2PC_MM_FN int d2pc_map_ray_next(d2pc_map_ray *r) {
  if (++r->steps > kD2pcMapRayMaxSteps) return 0;
  int dim;
  if (r->tmax[0] < r->tmax[1]) dim = r->tmax[0] < r->tmax[2] ? 0 : 2;
  else dim = r->tmax[1] < r->tmax[2] ? 1 : 2;
  r->key[dim] = (uint16_t)(r->key[dim] + r->step[dim]);
  r->tmax[dim] = D2PC_MM_DADD(r->tmax[dim], r->tdelta[dim]);
  if (r->key[0] == r->end[0] && r->key[1] == r->end[1] && r->key[2] == r->end[2]) return 0;
  /* std::min(a, b) is (b < a) ? b : a */
  const double m01 = r->tmax[1] < r->tmax[0] ? r->tmax[1] : r->tmax[0];
  const double dist = r->tmax[2] < m01 ? r->tmax[2] : m01;
  return !(dist > r->length);
}

/* insertScan's end of the ray for point p from origin o: p itself (*hit = 1) when max_range < 0 or |p - o| <=
 * max_range, else o + normalized(p - o) * (float)max_range (*hit = 0: no occupied cell) */
D2PC_MM_FN void d2pc_map_ray_end(const float o[3], const float p[3], double max_range, float e[3], int *hit) {
  const float d[3] = {D2PC_MM_FSUB(p[0], o[0]), D2PC_MM_FSUB(p[1], o[1]), D2PC_MM_FSUB(p[2], o[2])};
  const double n = d2pc_map_norm(d[0], d[1], d[2]);
  if (max_range < 0.0 || n <= max_range) {
    *hit = 1;
    for (int i = 0; i < 3; ++i) e[i] = p[i];
    return;
  }
  *hit = 0;
  /* Vector3::normalize: divide by (float)norm when norm > 0 (here norm > max_range >= 0) */
  const float len = D2PC_MM_D2F(n), mr = D2PC_MM_D2F(max_range);
  for (int i = 0; i < 3; ++i) e[i] = D2PC_MM_FADD(o[i], D2PC_MM_FMUL(D2PC_MM_FDIV(d[i], len), mr));
}

/* Morton code of a key: bits interleaved z, y, x from bit 15 down (octomap's child order, x lowest) */
D2PC_MM_FN uint64_t d2pc_map_morton(uint16_t kx, uint16_t ky, uint16_t kz) {
  uint64_t m = 0;
  for (int b = 15; b >= 0; --b)
    m = (m << 3) | ((uint64_t)((kz >> b) & 1) << 2) | ((uint64_t)((ky >> b) & 1) << 1) | (uint64_t)((kx >> b) & 1);
  return m;
}

#endif /* D2PC_MAP_MATH_H_ */
