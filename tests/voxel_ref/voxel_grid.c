/* voxel_grid.c -- CPU reference of D2PC_FILTER_VOXEL (test infrastructure, not product code).
 *
 * pcl::VoxelGrid<pcl::PointXYZ>::applyFilter (PCL 1.7.2 - 1.12, downsample_all_data = true,
 * filter_limit_negative = false) restated step by step from the recipe in include/d2pc_b200.h, with the one
 * choice PCL leaves open fixed: the points of a voxel are summed in ascending point index (PCL's std::sort is not
 * stable).  Plain C, float32 arithmetic as written (built with -ffp-contract=off), a comparison sort on
 * (idx, point index) for the stable order. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
  int64_t idx;
  uint32_t point;
} entry;

static int cmp_entry(const void *a, const void *b) {
  const entry *x = (const entry *)a, *y = (const entry *)b;
  if (x->idx != y->idx) return x->idx < y->idx ? -1 : 1;
  return x->point < y->point ? -1 : (x->point > y->point);
}

/* cloud: n points of 16 bytes {x, y, z, pad}.  out: room for n points.  Returns the number of points written;
 * *is_dense receives the cloud's is_dense flag. */
size_t d2pc_voxel_ref(const float *cloud, size_t n, float leaf_x, float leaf_y, float leaf_z, uint32_t min_points,
                      int limit_field, double limit_min, double limit_max, float *out, int *is_dense) {
  const float inv[3] = {1.0f / leaf_x, 1.0f / leaf_y, 1.0f / leaf_z};
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  size_t n_in = 0;
  unsigned char *inc = (unsigned char *)malloc(n ? n : 1);
  for (size_t i = 0; i < n; ++i) {
    const float *p = cloud + 4 * i;
    int ok = isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]);
    if (ok && limit_field >= 0) {
      const double v = (double)p[limit_field];
      ok = !(v < limit_min || v > limit_max);
    }
    inc[i] = (unsigned char)ok;
    if (!ok) continue;
    ++n_in;
    for (int a = 0; a < 3; ++a) {
      if (p[a] < mn[a]) mn[a] = p[a];
      if (p[a] > mx[a]) mx[a] = p[a];
    }
  }
  *is_dense = 1;
  if (n_in == 0) {
    free(inc);
    return 0;
  }
  /* step 4: PCL's overflow guard (decided in double: exact for this comparison, defined for any span) */
  double prod = 1.0;
  for (int a = 0; a < 3; ++a) {
    const float span = (mx[a] - mn[a]) * inv[a];
    prod *= trunc((double)span) + 1.0;
  }
  int fallback = !(prod <= 2147483647.0);
  /* step 5, and where PCL's int arithmetic would overflow, the same fallback */
  int min_b[3] = {0, 0, 0};
  int64_t mul[3] = {1, 0, 0};
  double div[3], spanmax[3];
  for (int a = 0; a < 3 && !fallback; ++a) {
    const float lo = floorf(mn[a] * inv[a]), hi = floorf(mx[a] * inv[a]);
    if (!((double)lo >= -2147483648.0 && (double)hi < 2147483648.0)) {
      fallback = 1;
      break;
    }
    min_b[a] = (int)lo;
    div[a] = (double)hi - (double)lo + 1.0;
    spanmax[a] = (double)(hi - (float)min_b[a]);
  }
  if (!fallback && !(spanmax[0] + spanmax[1] * div[0] + spanmax[2] * div[0] * div[1] < 2147483647.0)) fallback = 1;
  if (fallback) {
    memcpy(out, cloud, n * 16);
    *is_dense = 0;
    free(inc);
    return n;
  }
  mul[1] = (int64_t)div[0];
  mul[2] = (int64_t)div[0] * (int64_t)div[1];
  /* step 6 */
  entry *e = (entry *)malloc(n_in * sizeof(entry));
  size_t k = 0;
  for (size_t i = 0; i < n; ++i) {
    if (!inc[i]) continue;
    const float *p = cloud + 4 * i;
    int64_t idx = 0;
    for (int a = 0; a < 3; ++a) {
      const int ijk = (int)(floorf(p[a] * inv[a]) - (float)min_b[a]);
      idx += (int64_t)ijk * mul[a];
    }
    e[k].idx = idx;
    e[k].point = (uint32_t)i;
    ++k;
  }
  free(inc);
  qsort(e, n_in, sizeof(entry), cmp_entry);
  /* steps 7-8 */
  size_t n_out = 0;
  for (size_t a = 0; a < n_in;) {
    size_t b = a + 1;
    while (b < n_in && e[b].idx == e[a].idx) ++b;
    if (b - a >= min_points) {
      float s[3] = {0.0f, 0.0f, 0.0f};
      for (size_t m = a; m < b; ++m)
        for (int c = 0; c < 3; ++c) s[c] += cloud[4 * (size_t)e[m].point + c];
      const float cnt = (float)(b - a);
      float *o = out + 4 * n_out++;
      o[0] = s[0] / cnt, o[1] = s[1] / cnt, o[2] = s[2] / cnt, o[3] = 1.0f;
    }
    a = b;
  }
  free(e);
  return n_out;
}
