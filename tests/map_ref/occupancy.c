/* occupancy.c -- the occupancy map recipe of include/d2pc_b200.h ("occupancy map") per ray, on the library's own
 * csrc/map_math.h (test infrastructure, not product code).  Compiled with -ffp-contract=off, so every operation of
 * map_math.h is one IEEE operation as on the device.
 *
 * d2pc_map_ray_ref: the cells one point contributes to a frame -- the free cells of its ray in DDA order and, when the
 * point is within max_range and its key valid, the occupied cell.
 * d2pc_map_rays_digest: the same for n (origin, point) pairs, reduced to (free cell count, FNV-1a hash of the free
 * keys, occupied key or ~0) per pair, for comparisons over millions of rays. */
#include <stddef.h>
#include <stdint.h>

#include "map_math.h"

/* returns the number of free cells (all of them are counted; at most cap are written to keys, 3 per cell) */
uint32_t d2pc_map_ray_ref(const float o[3], const float p[3], double res, double max_range, uint16_t *keys,
                          uint32_t cap, uint16_t hit_key[3], int *hit_valid) {
  const double rf = 1.0 / res;
  *hit_valid = 0;
  if (!isfinite(p[0]) || !isfinite(p[1]) || !isfinite(p[2])) return 0;
  float e[3];
  int hit;
  d2pc_map_ray_end(o, p, max_range, e, &hit);
  uint32_t n = 0;
  d2pc_map_ray r;
  if (d2pc_map_ray_begin(&r, o, e, res, rf)) {
    do {
      if (n < cap)
        for (int a = 0; a < 3; ++a) keys[3 * n + a] = r.key[a];
      ++n;
    } while (d2pc_map_ray_next(&r));
  }
  if (hit && d2pc_map_key3(rf, p[0], p[1], p[2], hit_key)) *hit_valid = 1;
  return n;
}

static uint64_t fnv(uint64_t h, uint16_t v) {
  for (int b = 0; b < 2; ++b) h = (h ^ ((v >> (8 * b)) & 0xff)) * 0x100000001b3ull;
  return h;
}

/* pairs: n x 6 floats (ox, oy, oz, px, py, pz); out: n x 3 (count, hash, occupied key packed or ~0) */
void d2pc_map_rays_digest(const float *pairs, size_t n, double res, double max_range, uint64_t *out) {
  const double rf = 1.0 / res;
  for (size_t i = 0; i < n; ++i) {
    const float *o = pairs + 6 * i, *p = pairs + 6 * i + 3;
    uint64_t count = 0, h = 0xcbf29ce484222325ull, occ = ~0ull;
    if (isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2])) {
      float e[3];
      int hit;
      d2pc_map_ray_end(o, p, max_range, e, &hit);
      d2pc_map_ray r;
      if (d2pc_map_ray_begin(&r, o, e, res, rf)) {
        do {
          ++count;
          for (int a = 0; a < 3; ++a) h = fnv(h, r.key[a]);
        } while (d2pc_map_ray_next(&r));
      }
      uint16_t k[3];
      if (hit && d2pc_map_key3(rf, p[0], p[1], p[2], k))
        occ = (uint64_t)k[0] | ((uint64_t)k[1] << 16) | ((uint64_t)k[2] << 32);
    }
    out[3 * i] = count, out[3 * i + 1] = h, out[3 * i + 2] = occ;
  }
}

uint64_t d2pc_map_morton_ref(uint16_t kx, uint16_t ky, uint16_t kz) { return d2pc_map_morton(kx, ky, kz); }
