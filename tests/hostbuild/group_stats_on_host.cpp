// group_stats_on_host.cpp -- TEST HARNESS, not part of the product.
//
// Compiles the rules of samsim_b200/csrc/group_stats.cuh (member layout, depth regrid, final statistics) for the host,
// so that the no-GPU test stage can check them against the numpy reference (tests/test_group_stats_cpu.py).
#include <stdint.h>
#include <string.h>

#define __device__
#define __host__

#include "../../samsim_b200/csrc/group_stats.cuh"

using namespace samsim;

extern "C" {

// padded layout of a group assignment; copies it out when it fits `cap` entries, returns its length
int64_t gsh_layout(int64_t ncol, int32_t ngroup, const int32_t* group_of_col, int32_t* col, int32_t* info, int64_t cap,
                   int64_t* start, int32_t* lg) {
  const GsLayout L = gs_layout(ncol, ngroup, group_of_col);
  if (L.npad <= cap) {
    memcpy(col, L.col.data(), (size_t)L.npad * sizeof(int32_t));
    memcpy(info, L.info.data(), (size_t)L.npad * sizeof(int32_t));
    memcpy(start, L.start.data(), (size_t)ngroup * sizeof(int64_t));
    memcpy(lg, L.lg.data(), (size_t)ngroup * sizeof(int32_t));
  }
  return L.npad;
}

// layer (1-based) of each depth, 0 where the depth is below the column's ice; returns D_{n_active}
double gsh_regrid(const double* thick, int32_t n_active, const double* z, int32_t nz, int32_t* layer) {
  for (int j = 0; j < nz; j++) layer[j] = 0;
  return gs_regrid([&](int k) { return thick[k - 1]; }, n_active, z, nz, [&](int j, int k) { layer[j] = k; });
}

// mean and variance from count and the two tree sums
void gsh_finish(int32_t n, const double* count, const double* s, const double* m2, double* mean, double* var) {
  for (int q = 0; q < n; q++) {
    mean[q] = gs_mean(count[q], s[q]);
    var[q] = gs_variance(count[q], m2[q]);
  }
}

}  // extern "C"
