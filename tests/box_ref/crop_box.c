/* CPU reference of the crop box stage: the recipe of include/d2pc_b200.h, step by step (test infrastructure, not
 * product code).  Compiled with -ffp-contract=off, so every float operation below is rounded on its own.
 *
 *   size_t d2pc_box_ref(const float *pts, size_t n, const float mn[3], const float mx[3], const float t[12],
 *                       float *out)
 * pts: n points of 4 floats; t: row-major 3x4 [R | t]; out receives the kept points (4 floats each, unchanged) in
 * input order; returns their number. */
#include <math.h>
#include <stddef.h>
#include <string.h>

size_t d2pc_box_ref(const float *pts, size_t n, const float mn[3], const float mx[3], const float t[12], float *out) {
  size_t k = 0;
  for (size_t i = 0; i < n; ++i) {
    const float *p = pts + 4 * i;
    /* 1. only finite points take part */
    if (!(isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]))) continue;
    int in = 1;
    for (int a = 0; a < 3; ++a) {
      /* 2. l = T p, ((t0 x + t1 y) + t2 z) + t3 */
      const float *r = t + 4 * a;
      float l = r[0] * p[0];
      l = l + r[1] * p[1];
      l = l + r[2] * p[2];
      l = l + r[3];
      /* 3. inside when min <= l <= max (a NaN l is not) */
      if (!(mn[a] <= l && l <= mx[a])) in = 0;
    }
    /* 4. copied unchanged, in input order */
    if (in) memcpy(out + 4 * k++, p, 16);
  }
  return k;
}
