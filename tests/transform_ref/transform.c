/* CPU reference of the cloud transform stage: the recipe of include/d2pc_b200.h, step by step (test infrastructure,
 * not product code).  Compiled with -ffp-contract=off, so every float operation below is rounded on its own.
 *
 *   void d2pc_transform_ref(const float *pts, size_t n, const float m[12], float *out)
 * pts: n points of 4 floats; m: row-major 3x4 [A | t]; out receives n points of 4 floats in input order. */
#include <math.h>
#include <stddef.h>
#include <string.h>

void d2pc_transform_ref(const float *pts, size_t n, const float m[12], float *out) {
  for (size_t i = 0; i < n; ++i) {
    const float *p = pts + 4 * i;
    float *o = out + 4 * i;
    /* 2-3. every point starts as a copy of all 16 bytes (NaN payloads and the w word included) */
    memcpy(o, p, 16);
    /* 1. a point with finite x, y and z: row a = ((m0 x + m1 y) + m2 z) + m3 */
    if (!(isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]))) continue;
    for (int a = 0; a < 3; ++a) {
      const float *r = m + 4 * a;
      float v = r[0] * p[0];
      v = v + r[1] * p[1];
      v = v + r[2] * p[2];
      v = v + r[3];
      o[a] = v;
    }
  }
}
