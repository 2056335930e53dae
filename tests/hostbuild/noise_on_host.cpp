// noise_on_host.cpp -- TEST HARNESS, not part of the product.
//
// Compiles the rules of samsim_b200/csrc/noise.cuh (Philox, the normal deviate, the recursion, the modes and the
// cursor rule) for the host, so that the no-GPU test stage can check them against the numpy reference
// (tests/stochastic_ref.py) and the GPU tests can check the device against them.
#include <stdint.h>

#define __device__
#define __host__

#include "../../samsim_b200/csrc/noise.cuh"

using namespace samsim;

extern "C" {

void nh_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
  for (int j = 0; j < 4; j++) out[j] = ctr[j];
  philox4x32_10(out, key[0], key[1]);
}

void nh_det_log(int64_t n, const double* x, double* out) {
  for (int64_t q = 0; q < n; q++) out[q] = det_log(x[q]);
}
void nh_det_cos(int64_t n, const double* x, double* out) {
  for (int64_t q = 0; q < n; q++) out[q] = det_cos(x[q]);
}
void nh_det_exp(int64_t n, const double* x, double* out) {
  for (int64_t q = 0; q < n; q++) out[q] = det_exp(x[q]);
}

// out[q*nrec + r] = z(rec0 + r) of streams[q]
void nh_normals(uint64_t seed, int32_t kind, int32_t n, const int32_t* streams, int32_t rec0, int32_t nrec, double* out) {
  for (int32_t q = 0; q < n; q++)
    for (int32_t r = 0; r < nrec; r++) out[(int64_t)q * nrec + r] = noise_normal(seed, kind, streams[q], rec0 + r);
}

// out[q*nrec + r] = e(rec0 + r) of streams[q], the pure function (a window from an empty cursor)
void nh_series(uint64_t seed, double sigma, double phi, int32_t kind, int32_t n, const int32_t* streams, int32_t rec0,
               int32_t nrec, double* out) {
  const NoiseKind nk = noise_kind(sigma, phi, SAMSIM_NOISE_ADDITIVE);
  for (int32_t q = 0; q < n; q++) {
    double ep = 0.0, ec = 0.0;
    double* o = out + (int64_t)q * nrec;
    noise_window(nk, seed, kind, streams[q], 0, rec0, rec0 + nrec - 1, ep, ec, [&](int32_t r, double e) { o[r - rec0] = e; });
  }
}

// One launch window first..last of the device's window kernel for n streams, from the cursor and the held state
// state[2q], state[2q+1]; out[q*(last-first+1) + r - first] = e(r).  Returns the new cursor.
int32_t nh_window(uint64_t seed, double sigma, double phi, int32_t kind, int32_t n, const int32_t* streams, int32_t cursor,
                  int32_t first, int32_t last, double* state, double* out) {
  const NoiseKind nk = noise_kind(sigma, phi, SAMSIM_NOISE_ADDITIVE);
  const int64_t len = (int64_t)last - first + 1;
  for (int32_t q = 0; q < n; q++) {
    double* o = out + q * len;
    noise_window(nk, seed, kind, streams[q], cursor, first, last, state[2 * q], state[2 * q + 1],
                 [&](int32_t r, double e) { o[r - first] = e; });
  }
  return noise_cursor_after(cursor, first, last);
}

// out[q] = the value v[q] perturbed by e[q] in `mode`
void nh_apply(int32_t mode, double sigma, double phi, int64_t n, const double* v, const double* e, double* out) {
  const NoiseKind nk = noise_kind(sigma, phi, mode);
  for (int64_t q = 0; q < n; q++) out[q] = noise_apply(nk, v[q], e[q]);
}

}  // extern "C"
