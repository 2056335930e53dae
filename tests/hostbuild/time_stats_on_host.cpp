// time_stats_on_host.cpp -- TEST HARNESS, not part of the product.
//
// Compiles the rules of samsim_b200/csrc/time_stats.cuh (Welford update, finalising, windows completed by a call) for
// the host, so that the no-GPU test stage can check them against the numpy reference (tests/test_time_stats_cpu.py).
#include <stdint.h>

#define __device__
#define __host__

#include "../../samsim_b200/csrc/time_stats.cuh"

using namespace samsim;

extern "C" {

// nq independent accumulators over nrec records: x[r*nq + q] enters where c[r*nq + q] != 0; out[q*5 + s]
void tsh_accumulate(int32_t nrec, int32_t nq, const double* x, const uint8_t* c, double* out) {
  for (int q = 0; q < nq; q++) {
    TsAcc a = ts_init();
    for (int r = 0; r < nrec; r++)
      if (c[(size_t)r * nq + q]) ts_update(a, x[(size_t)r * nq + q]);
    ts_finish(a, out + (size_t)q * SAMSIM_TS_NSTAT);
  }
}

int64_t tsh_records_in(int64_t i, int32_t n_time_out, int32_t i_time_out, int64_t nsteps) {
  return ts_records_in(i, n_time_out, i_time_out, nsteps);
}

int64_t tsh_windows_completed(int32_t records_per_window, int64_t in_window, int64_t nrec) {
  return ts_windows_completed(records_per_window, in_window, nrec);
}

}  // extern "C"
