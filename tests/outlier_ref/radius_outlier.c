/* radius_outlier.c -- CPU references of the radius outlier stage (test infrastructure, not product code).
 *
 * The recipe of include/d2pc_b200.h restated twice in plain C (built with -ffp-contract=off, so every float
 * operation below rounds on its own):
 *   d2pc_ror_brute  the rule literally: every pair, O(N^2);
 *   d2pc_ror_grid   the same answer from a uniform grid, fast enough for a 4K CROP cloud on one core.  Its grid is
 *                   deliberately not the GPU's: cells of c = max(r, 2^-64) * (1 + 2^-10) (doubled until every axis
 *                   has at most 2^20 cells), cell = floor((x - min) / c) with a division, three 21-bit fields in
 *                   the key.  The margin argument of csrc/radius_outlier.cu holds for it as well.
 * Both write the kept points, unchanged and in input order, to `out` and return how many there are. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static int finite3(const float *p) { return isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]); }

/* rule 3: FLANN's L2_Simple<float> */
static float dist2(const float *a, const float *b) {
  const float dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
  return (dx * dx + dy * dy) + dz * dz;
}

static size_t emit(const float *cloud, size_t n, const unsigned char *keep, float *out) {
  size_t k = 0;
  for (size_t i = 0; i < n; ++i)
    if (keep[i]) memcpy(out + 4 * k++, cloud + 4 * i, 16);
  return k;
}

size_t d2pc_ror_brute(const float *cloud, size_t n, double radius, uint32_t min_neighbors, float *out) {
  const double r2 = radius * radius;
  const uint64_t need = (uint64_t)min_neighbors + 1;
  unsigned char *keep = (unsigned char *)calloc(n ? n : 1, 1);
  for (size_t i = 0; i < n; ++i) {
    const float *p = cloud + 4 * i;
    if (!finite3(p)) continue;
    uint64_t cnt = 0;
    for (size_t j = 0; j < n && cnt < need; ++j) {
      const float *q = cloud + 4 * j;
      if (finite3(q) && (double)dist2(p, q) <= r2) ++cnt;
    }
    keep[i] = cnt >= need;
  }
  const size_t k = emit(cloud, n, keep, out);
  free(keep);
  return k;
}

typedef struct {
  uint64_t key;
  uint32_t idx;
} item;

static int cmp_item(const void *a, const void *b) {
  const item *x = (const item *)a, *y = (const item *)b;
  if (x->key != y->key) return x->key < y->key ? -1 : 1;
  return x->idx < y->idx ? -1 : (x->idx > y->idx);
}

#define AXIS_BITS 21
#define MAX_AXIS_CELLS (1u << 20) /* cells holding points; with the padding every field stays below 2^21 */

/* first position in [lo, hi) with key >= k */
static size_t lower(const item *it, size_t lo, size_t hi, uint64_t k) {
  while (lo < hi) {
    const size_t mid = lo + (hi - lo) / 2;
    if (it[mid].key < k) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

size_t d2pc_ror_grid(const float *cloud, size_t n, double radius, uint32_t min_neighbors, float *out) {
  const double r2 = radius * radius;
  const uint64_t need = (uint64_t)min_neighbors + 1;
  unsigned char *keep = (unsigned char *)calloc(n ? n : 1, 1);
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  size_t m = 0;
  for (size_t i = 0; i < n; ++i) {
    const float *p = cloud + 4 * i;
    if (!finite3(p)) continue;
    ++m;
    for (int a = 0; a < 3; ++a) {
      if (p[a] < mn[a]) mn[a] = p[a];
      if (p[a] > mx[a]) mx[a] = p[a];
    }
  }
  if (m == 0) {
    free(keep);
    return 0;
  }
  double c = fmax(radius, 0x1p-64) * (1.0 + 0x1p-10);
  for (;; c *= 2.0) {
    int ok = 1;
    for (int a = 0; a < 3; ++a) ok &= floor(((double)mx[a] - (double)mn[a]) / c) + 1.0 <= MAX_AXIS_CELLS;
    if (ok) break;
  }
  item *it = (item *)malloc(m * sizeof(item));
  size_t k = 0;
  for (size_t i = 0; i < n; ++i) {
    const float *p = cloud + 4 * i;
    if (!finite3(p)) continue;
    uint64_t key = 0;
    for (int a = 0; a < 3; ++a)
      key |= ((uint64_t)floor(((double)p[a] - (double)mn[a]) / c) + 1) << (AXIS_BITS * a);
    it[k].key = key;
    it[k].idx = (uint32_t)i;
    ++k;
  }
  qsort(it, m, sizeof(item), cmp_item);
  for (size_t s = 0; s < m; ++s) {
    const float *p = cloud + 4 * (size_t)it[s].idx;
    const uint64_t key = it[s].key;
    uint64_t cnt = 0;
    for (int dz = -1; dz <= 1 && cnt < need; ++dz)
      for (int dy = -1; dy <= 1 && cnt < need; ++dy) {
        /* the row (x - 1 .. x + 1, y + dy, z + dz): one contiguous key range (cells start at 1, so no borrow) */
        const uint64_t row = key + (uint64_t)(int64_t)dy * (1ull << AXIS_BITS) + (uint64_t)(int64_t)dz * (1ull << (2 * AXIS_BITS));
        const size_t lo = lower(it, 0, m, row - 1), hi = lower(it, lo, m, row + 2);
        for (size_t t = lo; t < hi && cnt < need; ++t)
          if ((double)dist2(p, cloud + 4 * (size_t)it[t].idx) <= r2) ++cnt;
      }
    keep[it[s].idx] = cnt >= need;
  }
  free(it);
  k = emit(cloud, n, keep, out);
  free(keep);
  return k;
}
