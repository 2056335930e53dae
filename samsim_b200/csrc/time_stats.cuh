// time_stats.cuh -- per-column time statistics over windows of S8 records (samsim_b200_set_time_stats).
//
// The rules that fix every bit of the result live here as plain functions, so that tests/hostbuild can compile them
// for the host: the Welford update of one record, the finalising of a window and the number of windows a
// samsim_b200_step call completes.  The regrid of a profile onto the depth grid and the variance are those of the
// group statistics (gs_regrid, gs_variance in group_stats.cuh).  The kernels that use them are in samsim_b200.cu.
//
// Accumulation.  Records enter in record order, each column and quantity on its own, starting from n = 0, mean = 0,
// M2 = 0, min = max = NaN:
//   n = n + 1;  d = x - mean;  mean = mean + d / n;  M2 = M2 + d * (x - mean);  min = fmin(min, x);  max = fmax(max, x)
// (compiled without contraction: -fmad=false on the device, -ffp-contract=off on the host).  fmin / fmax keep the
// earlier value of two equal ones, so +0.0 and -0.0 resolve the same way everywhere (ts_min, ts_max).
#pragma once

#include <math.h>
#include <stdint.h>

#include "group_stats.cuh"

#define SAMSIM_TS_NSTAT 5  // count, mean, variance, min, max

namespace samsim {

// one column and quantity of the window in progress
struct TsAcc {
  double n, mean, m2, mn, mx;
};

__host__ __device__ inline TsAcc ts_init() { return TsAcc{0.0, 0.0, 0.0, nan(""), nan("")}; }

// fmin / fmax with the tie fixed: a NaN accumulator takes x, a NaN x is skipped, and of two equal values (+0.0 and
// -0.0) the accumulator's stays
__host__ __device__ inline double ts_min(double m, double x) { return (x < m || m != m) ? x : m; }
__host__ __device__ inline double ts_max(double m, double x) { return (x > m || m != m) ? x : m; }

__host__ __device__ inline void ts_update(TsAcc& a, double x) {
  a.n = a.n + 1.0;
  const double d = x - a.mean;
  a.mean = a.mean + d / a.n;
  a.m2 = a.m2 + d * (x - a.mean);
  a.mn = ts_min(a.mn, x);
  a.mx = ts_max(a.mx, x);
}

// count, mean (NaN for count 0), variance (gs_variance: M2 / (n - 1), 0 for n = 1, NaN for n = 0), min, max (NaN for
// count 0: nothing replaced the initial NaN)
__host__ __device__ inline void ts_finish(const TsAcc& a, double out[SAMSIM_TS_NSTAT]) {
  out[0] = a.n;
  out[1] = (a.n > 0.0) ? a.mean : nan("");
  out[2] = gs_variance(a.n, a.m2);
  out[3] = a.mn;
  out[4] = a.mx;
}

// S8 records that `nsteps` steps write from the clock (i, n_time_out): the step to loop index 1 writes one, and then
// every (i_time_out + 1)-th step (mo_grotz.f90:340)
__host__ __device__ inline int64_t ts_records_in(int64_t i, int32_t n_time_out, int32_t i_time_out, int64_t nsteps) {
  const int64_t first = (i == 0) ? 1 : (int64_t)(i_time_out - n_time_out) + 1;
  return (nsteps < first) ? 0 : 1 + (nsteps - first) / ((int64_t)i_time_out + 1);
}

// windows that `nrec` more records complete, with `in_window` records already in the window in progress;
// records_per_window = 0: only samsim_b200_close_time_window closes a window
__host__ __device__ inline int64_t ts_windows_completed(int32_t records_per_window, int64_t in_window, int64_t nrec) {
  return (records_per_window > 0) ? (in_window + nrec) / records_per_window : 0;
}

}  // namespace samsim
