// detmath.h -- deterministic FP64 exp / log / pow / sin / cos.
//
// Why this exists.  The SAMSIM column timestep needs four transcendental
// functions: x**3.10 (permeability, mo_grav_drain.f90:104-106, mo_flush.f90:113-129,
// mo_flood.f90:73), x**1.5 (func_density mo_functions.f90:60, func_T_freeze :248),
// EXP (Beer law mo_heat_fluxes.f90:152-155, sub_turb_flux mo_functions.f90:359) and
// SIN (sub_test4, mo_testcase_specifics.f90:200).  The reference calls the compiler
// runtime (glibc libm); CUDA's libdevice versions differ from glibc in the last
// bit for some arguments, which would make a GPU column drift from a CPU column
// by ~1e-16 per call and flip layer-dynamics events after enough steps.
//
// Every function below is built from IEEE-754 correctly rounded operations only
// (+ - * / and fma), with no data-dependent library calls, so that the SAME
// source compiled by gcc (-ffp-contract=off) and by nvcc (-fmad=false) returns
// bit-identical results on the host and on sm_100a.  Accuracy is < 1 ulp
// (measured against glibc in tests/test_detmath.py), i.e. the same quality as the
// runtime the reference uses, but reproducible across CPU and GPU.
//
// Domain notes: det_pow is defined for x >= 0 and finite y (the only uses are
// x >= 0 with y in {1.5, 3.1}); det_sin/det_cos use a 3-term Cody-Waite reduction
// that is accurate for |x| < 1e5 (the model passes phases below 30).
#ifndef SAMSIM_B200_DETMATH_H
#define SAMSIM_B200_DETMATH_H

#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define DM_HD __host__ __device__ __forceinline__
// the public entry points are single out-of-line copies on the device: the step kernel calls them from many
// sites and its instruction footprint, not call overhead, is what stalls the warps (I-cache misses)
#define DM_API __host__ __device__ __noinline__
#else
#define DM_HD static inline
#define DM_API static inline
#include <string.h>
#endif

DM_HD int64_t dm_bits(double x) {
#if defined(__CUDA_ARCH__)
  return __double_as_longlong(x);
#else
  int64_t b;
  memcpy(&b, &x, sizeof b);
  return b;
#endif
}

DM_HD double dm_from_bits(int64_t b) {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double(b);
#else
  double x;
  memcpy(&x, &b, sizeof x);
  return x;
#endif
}

// 2^k for k in [-1022, 1023]
DM_HD double dm_pow2i(int k) { return dm_from_bits((int64_t)(k + 1023) << 52); }

// p * 2^k with a single rounding (p in [0.5, 2]), correct into the subnormal range.
DM_HD double dm_scale2(double p, int k) {
  if (k > 1023) {
    if (k > 2000) k = 2000;
    return (p * dm_pow2i(1023)) * dm_pow2i(k - 1023);
  }
  if (k < -1021) {
    if (k < -2000) k = -2000;
    int k1 = k / 2;
    return (p * dm_pow2i(k1)) * dm_pow2i(k - k1);
  }
  return p * dm_pow2i(k);
}

// exp(r) for |r| <= 0.36 (after reduction); rl is a small correction added to r.
DM_HD double dm_exp_kernel(double r, double rl) {
  // Taylor coefficients 1/n!, n = 2..13, Horner with fma.
  double q = 1.6059043836821613e-10;            // 1/13!
  q = fma(q, r, 2.08767569878681e-09);          // 1/12!
  q = fma(q, r, 2.505210838544172e-08);         // 1/11!
  q = fma(q, r, 2.755731922398589e-07);         // 1/10!
  q = fma(q, r, 2.7557319223985893e-06);        // 1/9!
  q = fma(q, r, 2.48015873015873e-05);          // 1/8!
  q = fma(q, r, 0.0001984126984126984);         // 1/7!
  q = fma(q, r, 0.001388888888888889);          // 1/6!
  q = fma(q, r, 0.008333333333333333);          // 1/5!
  q = fma(q, r, 0.041666666666666664);          // 1/4!
  q = fma(q, r, 0.16666666666666666);           // 1/3!
  q = fma(q, r, 0.5);                           // 1/2!
  // exp(r+rl) = 1 + r + r^2 q + rl (1 + r) to first order in rl
  double r2q = (r * r) * q;
  double t = r2q + fma(rl, r, rl);
  return 1.0 + (r + t);
}

#define DM_LN2_HI 6.93147180369123816490e-01  /* 0x3fe62e42fee00000, 33 significant bits */
#define DM_LN2_LO 1.90821492927058770002e-10  /* ln2 - DM_LN2_HI */
#define DM_INV_LN2 1.44269504088896338700e+00

// exp(xh + xl), |xl| << |xh|
DM_HD double dm_exp2part(double xh, double xl) {
  if (xh > 709.8) return dm_from_bits(0x7ff0000000000000LL);  // +inf
  if (xh < -745.2) return 0.0;
  double kd = rint(xh * DM_INV_LN2);
  int k = (int)kd;
  double r = fma(-kd, DM_LN2_HI, xh);   // exact: kd has <= 11 bits, LN2_HI 33 bits
  double rl = fma(-kd, DM_LN2_LO, xl);
  // fold the low part into r, keep the residual
  double rs = r + rl;
  double rr = rl - (rs - r);
  double p = dm_exp_kernel(rs, rr);
  return dm_scale2(p, k);
}

DM_API double det_exp(double x) {
  if (x != x) return x;
  return dm_exp2part(x, 0.0);
}

// log(x) as an unevaluated sum hi + lo, x > 0 finite.  Relative error ~2^-62.
DM_HD void dm_log2part(double x, double* hi, double* lo) {
  int e = 0;
  int64_t b = dm_bits(x);
  if (b < 0x0010000000000000LL) {  // subnormal: renormalise
    x = x * 18014398509481984.0;   // 2^54
    b = dm_bits(x);
    e = -54;
  }
  e += (int)(b >> 52) - 1023;
  int64_t mant = b & 0x000fffffffffffffLL;
  double m = dm_from_bits(mant | 0x3ff0000000000000LL);  // [1, 2)
  if (m > 1.4142135623730951) {
    m = m * 0.5;
    e += 1;
  }
  // s = (m-1)/(m+1) in double-double; m-1 is exact.
  double num = m - 1.0;
  double dh = m + 1.0;
  double dl = (m - (dh - 1.0));  // exact: two-sum tail (|m| >= |1| not required for these magnitudes, dh-1 exact)
  double sh = num / dh;
  double rem = fma(-sh, dh, num);
  rem = fma(-sh, dl, rem);
  double sl = rem / dh;
  // log(m) = 2 s + 2 s^3 (1/3 + s^2/5 + s^4/7 + ...)
  double z = sh * sh;
  double q = 0.07407407407407407;          // 2/27
  q = fma(q, z, 0.08);                     // 2/25
  q = fma(q, z, 0.08695652173913043);      // 2/23
  q = fma(q, z, 0.09523809523809523);      // 2/21
  q = fma(q, z, 0.10526315789473684);      // 2/19
  q = fma(q, z, 0.11764705882352941);      // 2/17
  q = fma(q, z, 0.13333333333333333);      // 2/15
  q = fma(q, z, 0.15384615384615385);      // 2/13
  q = fma(q, z, 0.18181818181818182);      // 2/11
  q = fma(q, z, 0.2222222222222222);       // 2/9
  q = fma(q, z, 0.2857142857142857);       // 2/7
  q = fma(q, z, 0.4);                      // 2/5
  q = fma(q, z, 0.6666666666666666);       // 2/3
  double tail = (sh * z) * q;              // 2 s^3 (...)
  // assemble: e*ln2_hi (exact) + 2*sh + [2*sl + tail + e*ln2_lo]
  double ed = (double)e;
  double a = ed * DM_LN2_HI;               // exact (|e| < 2^11, LN2_HI has 33 bits)
  double bterm = 2.0 * sh;
  double small = fma(ed, DM_LN2_LO, fma(2.0, sl, tail));
  // two-sum a + bterm (|a| >= |bterm| or a == 0)
  double s1 = a + bterm;
  double t1 = (a == 0.0) ? 0.0 : (bterm - (s1 - a));
  double l = t1 + small;
  double h = s1 + l;
  *lo = l - (h - s1);
  *hi = h;
}

DM_API double det_log(double x) {
  if (x != x || x < 0.0) return dm_from_bits(0x7ff8000000000000LL);
  if (x == 0.0) return dm_from_bits((int64_t)0xfff0000000000000ULL);
  if (dm_bits(x) == 0x7ff0000000000000LL) return x;
  double h, l;
  dm_log2part(x, &h, &l);
  return h + l;
}

// x**y for x >= 0.  pow(0, y>0) = 0, pow(x, 0) = 1.
DM_API double det_pow(double x, double y) {
  if (y == 0.0) return 1.0;
  if (x != x || y != y || x < 0.0) return dm_from_bits(0x7ff8000000000000LL);
  if (x == 0.0) return (y > 0.0) ? 0.0 : dm_from_bits(0x7ff0000000000000LL);
  if (dm_bits(x) == 0x7ff0000000000000LL) return (y > 0.0) ? x : 0.0;
  double lh, ll;
  dm_log2part(x, &lh, &ll);
  // (ph + pl) = y * (lh + ll)
  double ph = y * lh;
  double pl = fma(y, lh, -ph);
  pl = fma(y, ll, pl);
  return dm_exp2part(ph, pl);
}

// ---- inverse permeability, from below ----------------------------------------
// A lower bound of 1 / perm with perm = 1e-17 * det_pow(1000*|psi_l|, 3.10) (mo_grav_drain.f90:104-106), for the
// gravity-drainage bound that rules out layers without evaluating det_pow (physics.cuh, grav_drain).  No division:
// log2 of the mantissa by a degree-8 polynomial in m-1 on [sqrt(1/2), sqrt(2)), 2^f by a degree-6 polynomial on
// [-1/2, 1/2] (Chebyshev fits; together < 1e-7 relative, measured by tests/test_perm_bound_cpu.py), then the result
// is lowered by DM_PERM_SLACK.  Where 1/perm is a normal double the result r satisfies
//     (1 - 2*DM_PERM_SLACK) / perm  <=  r  <  (1 - DM_PERM_SLACK/2) / perm .
// Ends: psi_l = 0 gives +inf (= 1/0); 1000|psi_l| < 2^-256 gives 2^790 (1/perm > 2^849 there); 1000|psi_l| > 2^256
// gives 0; NaN and +-inf give NaN, which the caller treats like any non-finite bound (the layer is evaluated exactly).
#define DM_PERM_SLACK 1.52587890625e-05  /* 2^-16 */
DM_HD double dm_perm_inv_lo(double psi_l) {
  const double x = 1000.0 * fabs(psi_l);
  if (!(x <= 1.157920892373162e+77)) return (x != x || x > 1.7976931348623157e+308) ? dm_from_bits(0x7ff8000000000000LL) : 0.0;
  if (x < 8.636168555094445e-78) return (x == 0.0) ? dm_from_bits(0x7ff0000000000000LL) : dm_pow2i(790);  // 2^-256
  const int64_t b = dm_bits(x);
  int e = (int)(b >> 52) - 1023;
  double m = dm_from_bits((b & 0x000fffffffffffffLL) | 0x3ff0000000000000LL);  // [1, 2)
  if (m > 1.4142135623730951) {
    m = m * 0.5;
    e += 1;
  }
  const double u = m - 1.0;                 // exact
  double p = 0.12453901975427666;           // log2(1+u)/u
  p = fma(p, u, -0.2048054494423592);
  p = fma(p, u, 0.21508739257218026);
  p = fma(p, u, -0.23924569897150472);
  p = fma(p, u, 0.28800520316499323);
  p = fma(p, u, -0.3606933098145126);
  p = fma(p, u, 0.4809079378408423);
  p = fma(p, u, -0.7213474398355846);
  p = fma(p, u, 1.4426950148397704);
  const double t = -3.10 * ((double)e + u * p);  // log2(1/x^3.10), |t| < 800
  const double n = rint(t);
  const double f = t - n;                   // exact, |f| <= 1/2
  double q = 0.00015465312336038613;        // 2^f
  q = fma(q, f, 0.001339527980035732);
  q = fma(q, f, 0.00961803994572486);
  q = fma(q, f, 0.05550340680745591);
  q = fma(q, f, 0.24022651101313985);
  q = fma(q, f, 0.6931472000626802);
  q = fma(q, f, 0.9999999999718431);
  return 1e17 * ((q * (1.0 - DM_PERM_SLACK)) * dm_pow2i((int)n));
}

// ---- sin / cos ------------------------------------------------------------
#define DM_PIO2_1 1.57079632673412561417e+00 /* first 33 bits of pi/2 */
#define DM_PIO2_2 6.07710050630396597660e-11 /* second 33 bits */
#define DM_PIO2_3 2.02226624871116645580e-21 /* third part: pi/2 - (PIO2_1 + PIO2_2) */
#define DM_2_OVER_PI 6.36619772367581382433e-01

DM_HD double dm_sin_kernel(double x, double xl) {
  double z = x * x;
  double r = 1.58969099521155010221e-10;
  r = fma(r, z, -2.50507602534068634195e-08);
  r = fma(r, z, 2.75573137070700676789e-06);
  r = fma(r, z, -1.98412698298579493134e-04);
  r = fma(r, z, 8.33333333332248946124e-03);
  double v = z * x;
  // x + v*(S1 + z r) + xl (1 - z/2)
  double s1 = -1.66666666666666324348e-01;
  return x - ((z * (0.5 * xl - v * r) - xl) - v * s1);
}

DM_HD double dm_cos_kernel(double x, double xl) {
  double z = x * x;
  double r = -1.13596475577881948265e-11;
  r = fma(r, z, 2.08757232129817482790e-09);
  r = fma(r, z, -2.75573143513906633035e-07);
  r = fma(r, z, 2.48015872894767294178e-05);
  r = fma(r, z, -1.38888888888741095749e-03);
  r = fma(r, z, 4.16666666666666019037e-02);
  double hz = 0.5 * z;
  double w = 1.0 - hz;
  return w + (((1.0 - w) - hz) + (z * (z * r) - x * xl));
}

DM_HD int dm_rem_pio2(double x, double* rh, double* rl) {
  double kd = rint(x * DM_2_OVER_PI);
  int k = (int)kd;
  double r = fma(-kd, DM_PIO2_1, x);  // exact for |kd| < 2^20
  double w = kd * DM_PIO2_2;
  double y0 = r - w;
  // recover the rounding of r - w and add the third term
  double t = (r - y0) - w;
  double w3 = fma(kd, DM_PIO2_3, -t);
  double y = y0 - w3;
  *rl = (y0 - y) - w3;
  *rh = y;
  return k;
}

DM_API double det_sin(double x) {
  if (x != x || fabs(x) > 1.0e5) return dm_from_bits(0x7ff8000000000000LL);
  double rh, rl;
  int k = dm_rem_pio2(x, &rh, &rl);
  switch (k & 3) {
    case 0: return dm_sin_kernel(rh, rl);
    case 1: return dm_cos_kernel(rh, rl);
    case 2: return -dm_sin_kernel(rh, rl);
    default: return -dm_cos_kernel(rh, rl);
  }
}

DM_API double det_cos(double x) {
  if (x != x || fabs(x) > 1.0e5) return dm_from_bits(0x7ff8000000000000LL);
  double rh, rl;
  int k = dm_rem_pio2(x, &rh, &rl);
  switch (k & 3) {
    case 0: return dm_cos_kernel(rh, rl);
    case 1: return -dm_sin_kernel(rh, rl);
    case 2: return -dm_cos_kernel(rh, rl);
    default: return dm_sin_kernel(rh, rl);
  }
}

#endif  // SAMSIM_B200_DETMATH_H
