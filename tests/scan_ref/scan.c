/* CPU reference of the laser scan stage: the recipe of include/d2pc_b200.h, step by step (test infrastructure, not
 * product code).  range and angle come from the library's own csrc/scan_math.h, the one source the kernel compiles
 * too; the binning below restates the header's rules independently of csrc/laser_scan.cu.  Compiled with
 * -ffp-contract=off, so every operation is rounded on its own.
 *
 *   uint32_t d2pc_laser_scan_ref(const float *pts, size_t n_pts, const double prm[8], int use_inf, float *ranges,
 *                                uint32_t cap)
 * pts: n_pts points of 4 floats; prm = {min_height, max_height, angle_min, angle_max, angle_increment, range_min,
 * range_max, inf_epsilon}.  Returns the number of ranges n and writes the first min(n, cap) of them.
 *   double d2pc_scan_angle_ref(double y, double x), double d2pc_scan_range_ref(float x, float y): the shared math.
 *   void d2pc_scan_math_ref(const float *x, const float *y, size_t n, double *r, double *a): both over arrays. */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#include "scan_math.h"

double d2pc_scan_angle_ref(double y, double x) { return d2pc_scan_angle(y, x); }
double d2pc_scan_range_ref(float x, float y) { return d2pc_scan_range(x, y); }
void d2pc_scan_math_ref(const float *x, const float *y, size_t n, double *r, double *a) {
  for (size_t i = 0; i < n; ++i) r[i] = d2pc_scan_range(x[i], y[i]), a[i] = d2pc_scan_angle((double)y[i], (double)x[i]);
}

uint32_t d2pc_laser_scan_ref(const float *pts, size_t n_pts, const double prm[8], int use_inf, float *ranges,
                             uint32_t cap) {
  const double min_height = prm[0], max_height = prm[1], range_min = prm[5], range_max = prm[6];
  /* the message's float fields */
  const float angle_min = (float)prm[2], angle_max = (float)prm[3], angle_increment = (float)prm[4];
  const float range_max_f = (float)range_max;
  /* n in float arithmetic */
  const float span = angle_max - angle_min;
  const float q = span / angle_increment;
  const uint32_t n = (uint32_t)ceilf(q);
  const float init = use_inf ? INFINITY : (float)((double)range_max_f + prm[7]);
  for (uint32_t k = 0; k < n && k < cap; ++k) ranges[k] = init;
  for (size_t i = 0; i < n_pts; ++i) {
    const float x = pts[4 * i], y = pts[4 * i + 1], z = pts[4 * i + 2];
    if (isnan(x) || isnan(y) || isnan(z)) continue;
    if ((double)z > max_height || (double)z < min_height) continue;
    const double r = d2pc_scan_range(x, y);
    if (r < range_min || r > range_max) continue;
    const double a = d2pc_scan_angle((double)y, (double)x);
    if (a < (double)angle_min || a > (double)angle_max) continue;
    const int k = (int)((a - (double)angle_min) / (double)angle_increment);
    if ((uint32_t)k >= n) continue;
    const float fr = (float)r;
    /* the bin's value is the least (float)r of its points and the initial value */
    if (k < (int)cap && fr < ranges[k]) ranges[k] = fr;
  }
  return n;
}
