/* scan_math.h -- range(x, y) and angle(y, x) of the laser scan stage (include/d2pc_b200.h, "laser scan"), one source
 * for the CUDA kernel (csrc/laser_scan.cu) and the C reference (tests/scan_ref/scan.c), so the two meet byte for byte.
 *
 * Both are built only from IEEE-754 double add, sub, mul, div, sqrt and fma, each rounded to nearest on its own:
 * explicit __d*_rn / __fma_rn on the device, plain operators plus fma() on the host, where the file must be compiled
 * with -ffp-contract=off.  Neither CUDA's atan2 (not reproducible on the CPU) nor libm's (not on the device) is used.
 *
 *   d2pc_scan_range(x, y) = sqrt(x*x + y*y) for float x, y widened to double: the two products are exact, then one
 *       rounded add and a correctly rounded sqrt, so the result is within 1 ulp of the exact hypot.
 *   d2pc_scan_angle(y, x) = atan2(y, x) with C99's special values (signed zeros, +-pi, +-pi/2, +-pi/4, +-3pi/4 for
 *       the zero and infinite cases).  For float inputs the result is within 1 ulp of the exact atan2
 *       (tests/test_oracle_laser_scan.py measures it against mpmath at 60 digits).  The recipe:
 *         1. t = min(|x|, |y|) / max(|x|, |y|) in [0, 1], and the division's exact residual t_lo = fma(-t, den, num) / den;
 *         2. the nearest breakpoint c = k/8 (k = 0..8) and the reduced argument u = (t - c) / (1 + t*c), |u| <= 1/16,
 *            with t_lo / (1 + t*c) carried beside it;
 *         3. atan(t) = atan(c) + atan(u), atan(c) a double-double table, atan(u) = u + u^3 * P(u^2) with the Taylor
 *            series to u^15 (truncation error below 2^-64 of u);
 *         4. the octant: theta = C + s * atan(t) with (C, s) = (0, +1), (pi/2, -1), (pi, -1) or (pi/2, +1) for
 *            |y| <= |x|, x >= 0 / |y| > |x|, x >= 0 / |y| <= |x|, x < 0 / |y| > |x|, x < 0; the large terms are
 *            summed with error-free two-sums, so theta is rounded once;
 *         5. the sign of y.
 * How this differs from glibc's hypot and atan2: both glibc functions are also within 1 ulp, so the two can return
 * different doubles (usually 1 ulp apart) for some inputs.  A scan sees that only for a point whose range lies
 * within a few ulp of range_min / range_max or whose angle lies within a few ulp of a bin edge or of the angle
 * limits; everywhere else both pick the same bin and the same float range. */
#ifndef D2PC_SCAN_MATH_H_
#define D2PC_SCAN_MATH_H_

#include <math.h>

#if defined(__CUDACC__)
#define D2PC_SM_FN static __host__ __device__ __forceinline__
#else
#define D2PC_SM_FN static inline
#endif

#if defined(__CUDA_ARCH__)
#define D2PC_SM_ADD(a, b) __dadd_rn((a), (b))
#define D2PC_SM_SUB(a, b) __dsub_rn((a), (b))
#define D2PC_SM_MUL(a, b) __dmul_rn((a), (b))
#define D2PC_SM_DIV(a, b) __ddiv_rn((a), (b))
#define D2PC_SM_SQRT(a) __dsqrt_rn(a)
#define D2PC_SM_FMA(a, b, c) __fma_rn((a), (b), (c))
#else
#define D2PC_SM_ADD(a, b) ((a) + (b))
#define D2PC_SM_SUB(a, b) ((a) - (b))
#define D2PC_SM_MUL(a, b) ((a) * (b))
#define D2PC_SM_DIV(a, b) ((a) / (b))
#define D2PC_SM_SQRT(a) sqrt(a)
#define D2PC_SM_FMA(a, b, c) fma((a), (b), (c))
#endif

/* sqrt(x*x + y*y) for float inputs */
D2PC_SM_FN double d2pc_scan_range(float x, float y) {
  const double dx = (double)x, dy = (double)y;
  return D2PC_SM_SQRT(D2PC_SM_ADD(D2PC_SM_MUL(dx, dx), D2PC_SM_MUL(dy, dy)));
}

/* error-free a + b = *s + *e (Knuth's two-sum, six rounded operations) */
D2PC_SM_FN void d2pc_scan_two_sum(double a, double b, double *s, double *e) {
  const double t = D2PC_SM_ADD(a, b);
  const double bv = D2PC_SM_SUB(t, a);
  const double av = D2PC_SM_SUB(t, bv);
  *s = t;
  *e = D2PC_SM_ADD(D2PC_SM_SUB(a, av), D2PC_SM_SUB(b, bv));
}

/* atan(k/8), k = 0..8, as hi + lo (mpmath, 60 digits).  The device reads its copy through the read-only cache
 * (a table indexed per lane would otherwise live on the thread's stack). */
#define D2PC_SCAN_ATAN_HI                                                                                          \
  {0x0.0p+0, 0x1.fd5ba9aac2f6ep-4, 0x1.f5b75f92c80ddp-3, 0x1.6f61941e4def1p-2, 0x1.dac670561bb4fp-2,            \
   0x1.1e00babdefeb4p-1, 0x1.4978fa3269ee1p-1, 0x1.700a7c5784634p-1, 0x1.921fb54442d18p-1}
#define D2PC_SCAN_ATAN_LO                                                                                          \
  {0x0.0p+0, -0x1.cd37686760c17p-59, 0x1.8ab6e3cf7afbdp-57, -0x1.c63aae6f6e918p-56, 0x1.a2b7f222f65e2p-56,       \
   -0x1.928df287a668fp-58, 0x1.2419a87f2a458p-56, -0x1.8c34d25aadef6p-56, 0x1.1a62633145c07p-55}
#if defined(__CUDACC__)
static __device__ const double d2pc_scan_atan_hi_dev[9] = D2PC_SCAN_ATAN_HI;
static __device__ const double d2pc_scan_atan_lo_dev[9] = D2PC_SCAN_ATAN_LO;
#endif
static const double d2pc_scan_atan_hi_host[9] = D2PC_SCAN_ATAN_HI;
static const double d2pc_scan_atan_lo_host[9] = D2PC_SCAN_ATAN_LO;
#if defined(__CUDA_ARCH__)
#define D2PC_SCAN_ATAN_TABLE(t, k) __ldg((t##_dev) + (k))
#else
#define D2PC_SCAN_ATAN_TABLE(t, k) (t##_host)[k]
#endif

/* atan2(y, x) */
D2PC_SM_FN double d2pc_scan_angle(double y, double x) {
  const double pi_hi = 0x1.921fb54442d18p+1, pi_lo = 0x1.1a62633145c07p-53;
  const double pio2_hi = 0x1.921fb54442d18p+0, pio2_lo = 0x1.1a62633145c07p-54;
  const double pio4 = 0x1.921fb54442d18p-1, pi3o4 = 0x1.2d97c7f3321d2p+1;
  double r;
  if (x != x || y != y) return D2PC_SM_ADD(x, y);
  const int neg_y = signbit(y) != 0, neg_x = signbit(x) != 0;
  const double ax = neg_x ? -x : x, ay = neg_y ? -y : y;
  if (ay == 0.0) {
    r = neg_x ? pi_hi : 0.0; /* atan2(+-0, -0 or x < 0) = +-pi, atan2(+-0, +0 or x > 0) = +-0 */
  } else if (ax == 0.0) {
    r = pio2_hi;
  } else if (ax == INFINITY && ay == INFINITY) {
    r = neg_x ? pi3o4 : pio4;
  } else if (ax == INFINITY) {
    r = neg_x ? pi_hi : 0.0;
  } else if (ay == INFINITY) {
    r = pio2_hi;
  } else {
    /* 1. t = num / den in [0, 1] and its residual */
    const int swap = ay > ax;
    const double num = swap ? ax : ay, den = swap ? ay : ax;
    const double t = D2PC_SM_DIV(num, den);
    const double t_lo = D2PC_SM_DIV(D2PC_SM_FMA(-t, den, num), den);
    /* 2. breakpoint and reduced argument; t - c is exact (Sterbenz) */
    const int k = (int)D2PC_SM_ADD(D2PC_SM_MUL(t, 8.0), 0.5);
    const double c = D2PC_SM_MUL((double)k, 0.125);
    const double d = D2PC_SM_FMA(t, c, 1.0);
    const double u = D2PC_SM_DIV(D2PC_SM_SUB(t, c), d);
    const double u_lo = D2PC_SM_DIV(t_lo, d);
    /* 3. atan(u) - u = u^3 * P(u^2) */
    const double z = D2PC_SM_MUL(u, u);
    double p = -0x1.1111111111111p-4;           /* -1/15 */
    p = D2PC_SM_FMA(p, z, 0x1.3b13b13b13b14p-4);  /*  1/13 */
    p = D2PC_SM_FMA(p, z, -0x1.745d1745d1746p-4); /* -1/11 */
    p = D2PC_SM_FMA(p, z, 0x1.c71c71c71c71cp-4);  /*  1/9 */
    p = D2PC_SM_FMA(p, z, -0x1.2492492492492p-3); /* -1/7 */
    p = D2PC_SM_FMA(p, z, 0x1.999999999999ap-3);  /*  1/5 */
    p = D2PC_SM_FMA(p, z, -0x1.5555555555555p-2); /* -1/3 */
    p = D2PC_SM_MUL(D2PC_SM_MUL(u, z), p);
    /* 4. theta = C + s * (atan_hi[k] + u + (atan_lo[k] + u_lo + p)) */
    double c_hi, c_lo, s;
    if (!swap && !neg_x) c_hi = 0.0, c_lo = 0.0, s = 1.0;
    else if (swap && !neg_x) c_hi = pio2_hi, c_lo = pio2_lo, s = -1.0;
    else if (!swap) c_hi = pi_hi, c_lo = pi_lo, s = -1.0;
    else c_hi = pio2_hi, c_lo = pio2_lo, s = 1.0;
    double h1, e1, h2, e2;
    d2pc_scan_two_sum(c_hi, D2PC_SM_MUL(s, D2PC_SCAN_ATAN_TABLE(d2pc_scan_atan_hi, k)), &h1, &e1);
    d2pc_scan_two_sum(h1, D2PC_SM_MUL(s, u), &h2, &e2);
    const double tail = D2PC_SM_ADD(D2PC_SM_ADD(D2PC_SCAN_ATAN_TABLE(d2pc_scan_atan_lo, k), u_lo), p);
    const double lo = D2PC_SM_ADD(D2PC_SM_ADD(e1, e2), D2PC_SM_FMA(s, tail, c_lo));
    r = D2PC_SM_ADD(h2, lo);
  }
  /* 5. the sign of y */
  return neg_y ? -r : r;
}

#endif /* D2PC_SCAN_MATH_H_ */
