/* projected_map.c -- the projected 2-D map recipe of include/d2pc_b200.h in plain C (test infrastructure, not product
 * code), per voxel the way csrc/occupancy.cu computes it: the known voxels in Morton order (d2pc_occupancy_voxels'
 * output), each voxel's leaf level lambda from its aligned ranges (octomap_msg.c's test), then each voxel's leaf
 * extent into the min / max, the padding and the keys on the host side, and each voxel's leaf height test and value
 * into its own cell.  Keys, Morton codes, getNodeSize and keyToCoord are the library's csrc/map_math.h. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "map_math.h"

/* keys packed kx | ky << 16 | kz << 32 in Morton order, log-odds as float bits.  Returns 0 with the grid's size and
 * origin (width = height = 0 for n = 0), -3 when a padded corner has no key, -6 when memory runs out.  The cells are
 * written when cells is not NULL and cap >= width * height. */
int d2pc_projected_map_ref(const uint64_t *keys, const uint32_t *lo, size_t n, double res, float occ_thres,
                           double min_z, double max_z, double min_x_size, double min_y_size, int8_t *cells,
                           uint64_t cap, uint32_t *width, uint32_t *height, double origin[2]) {
  *width = *height = 0;
  origin[0] = origin[1] = 0.0;
  if (n == 0) return 0;
  uint64_t *m = malloc(n * 8);
  uint32_t *D = malloc(n * 4);
  uint8_t *lam = malloc(n);
  int rc = 0;
  if (!m || !D || !lam) {
    rc = -6;
    goto done;
  }
  for (size_t i = 0; i < n; ++i) {
    m[i] = d2pc_map_morton((uint16_t)keys[i], (uint16_t)(keys[i] >> 16), (uint16_t)(keys[i] >> 32));
    D[i] = i ? D[i - 1] + (lo[i] != lo[i - 1]) : 0;
  }
  for (size_t i = 0; i < n; ++i) {
    lam[i] = 16;
    for (int L = 15; L >= 0; --L) {
      const uint64_t size = 1ull << (3 * (16 - L)), o = m[i] & (size - 1);
      if (size > n || o > i) break;
      const uint64_t a = i - o, b = a + size - 1;
      if (b >= n || m[a] != m[i] - o || m[b] != m[i] - o + size - 1 || D[a] != D[b]) break;
      lam[i] = (uint8_t)L;
    }
  }
  /* each voxel's leaf: lo = c - size / 2, hi = lo + size */
  double mn[3] = {DBL_MAX, DBL_MAX, DBL_MAX}, mx[3] = {-DBL_MAX, -DBL_MAX, -DBL_MAX};
  for (size_t i = 0; i < n; ++i) {
    const double size = d2pc_map_node_size(lam[i], res);
    for (int a = 0; a < 3; ++a) {
      const double l = d2pc_map_node_centre((uint16_t)(keys[i] >> (16 * a)), lam[i], res) - size / 2.0, h = l + size;
      if (l < mn[a]) mn[a] = l;
      if (h > mx[a]) mx[a] = h;
    }
  }
  const double half[2] = {0.5 * min_x_size, 0.5 * min_y_size};
  for (int a = 0; a < 2; ++a) {
    if (-half[a] < mn[a]) mn[a] = -half[a];
    if (mx[a] < half[a]) mx[a] = half[a];
  }
  uint16_t kmin[3], kmax[3];
  const double rf = 1.0 / res;
  if (!d2pc_map_key3(rf, (float)mn[0], (float)mn[1], (float)mn[2], kmin) ||
      !d2pc_map_key3(rf, (float)mx[0], (float)mx[1], (float)mx[2], kmax)) {
    rc = -3;
    goto done;
  }
  *width = (uint32_t)(kmax[0] - kmin[0]) + 1u;
  *height = (uint32_t)(kmax[1] - kmin[1]) + 1u;
  for (int a = 0; a < 2; ++a) origin[a] = (double)(float)d2pc_map_centre(kmin[a], res) - res * 0.5;
  const uint64_t cells_n = (uint64_t)*width * *height;
  if (!cells || cap < cells_n) goto done;
  memset(cells, 0, cells_n); /* codes: 1 free, 2 occupied */
  for (size_t i = 0; i < n; ++i) {
    const double h = d2pc_map_node_size(lam[i], res) / 2.0;
    const double cz = d2pc_map_node_centre((uint16_t)(keys[i] >> 32), lam[i], res);
    if (!(cz + h > min_z && cz - h < max_z)) continue;
    float v;
    memcpy(&v, &lo[i], 4);
    const uint64_t at = (uint64_t)((uint16_t)(keys[i] >> 16) - kmin[1]) * *width + ((uint16_t)keys[i] - kmin[0]);
    cells[at] |= (int8_t)(v >= occ_thres ? 2 : 1);
  }
  for (uint64_t j = 0; j < cells_n; ++j) cells[j] = (int8_t)(cells[j] & 2 ? 100 : cells[j] ? 0 : -1);
done:
  free(m), free(D), free(lam);
  return rc;
}
