// correlated_noise_on_host.cpp -- TEST HARNESS, not part of the product.
//
// Compiles the rules of the correlated stochastic forcing in samsim_b200/csrc/noise.cuh (the argument rules, the
// Cholesky factor, the four-kind basis window and the column mix) for the host, so that the no-GPU test stage can check
// them against the numpy reference (tests/correlated_ref.py) and the GPU tests can check the device against them.  The
// single-stream rules are those of noise_on_host.cpp.
#include <stdint.h>
#include <string.h>

#define __device__
#define __host__

#include "../../samsim_b200/csrc/noise.cuh"

using namespace samsim;

extern "C" {

// noise_check: 0 for a valid setting, else 1 with the message in msg[256]; single, on and L as noise_check gives them
int32_t nh_check(const double* sigma, const double* phi, const int32_t* mode, const double* corr, int32_t nmix,
                 int64_t ncol, const int32_t* basis, const double* weight, int32_t* on_single, double* L, char* msg) {
  bool on = false, single = false;
  NoiseCorr nc;
  const char* bad = noise_check(sigma, phi, mode, corr, nmix, ncol, basis, weight, on, single, nc);
  msg[0] = 0;
  if (bad) {
    strncpy(msg, bad, 255);
    msg[255] = 0;
    return 1;
  }
  on_single[0] = on;
  on_single[1] = single;
  for (int q = 0; q < 16; q++) L[q] = nc.L[q];
  return 0;
}

// L of corr; returns 0 when corr is not positive definite
int32_t nh_cholesky(const double* corr, double* L) { return noise_cholesky(corr, L) ? 1 : 0; }

static NoiseCorr host_corr(const double* corr) {
  NoiseCorr nc = {};
  if (corr) {
    for (int i = 0; i < 4; i++)
      for (int j = 0; j < 4; j++) nc.on = nc.on || (i != j && corr[i * 4 + j] != 0.0);
    noise_cholesky(corr, nc.L);
  }
  return nc;
}

// One launch window first..last of samsim_noise_basis_kernel for n basis ids (corr NULL = the identity), from the
// cursor and the held state[(q*4 + k)*2 + {0, 1}]; out[(q*4 + k)*(last-first+1) + r - first] = E_k(r).  Returns the
// new cursor; cursor 0 gives the pure function.
int32_t nh_basis_window(uint64_t seed, const double* sigma, const double* phi, const double* corr, int32_t n,
                        const int32_t* ids, int32_t cursor, int32_t first, int32_t last, double* state, double* out) {
  NoiseKind nk[4];
  for (int k = 0; k < 4; k++) nk[k] = noise_kind(sigma[k], phi[k], SAMSIM_NOISE_ADDITIVE);
  const NoiseCorr nc = host_corr(corr);
  const int64_t len = (int64_t)last - first + 1;
  for (int32_t q = 0; q < n; q++) {
    double ep[4], ec[4];
    for (int k = 0; k < 4; k++) {
      ep[k] = state[(q * 4 + k) * 2];
      ec[k] = state[(q * 4 + k) * 2 + 1];
    }
    noise_basis_window(nk, nc, seed, ids[q], cursor, first, last, ep, ec, [&](int32_t r, const double* E) {
      for (int k = 0; k < 4; k++) out[((int64_t)q * 4 + k) * len + r - first] = E[k];
    });
    for (int k = 0; k < 4; k++) {
      state[(q * 4 + k) * 2] = ep[k];
      state[(q * 4 + k) * 2 + 1] = ec[k];
    }
  }
  return noise_cursor_after(cursor, first, last);
}

// The column mix of samsim_noise_mix_kernel for one kind: idx[c*nmix + m] a row of E[nb][nrec] or -1, weight likewise.
// e[c*nrec + r] the mixed value (0 for a column with no entry), q[c] its sum of squared weights, any[c] whether it
// has an entry.
void nh_mix(int32_t ncol, int32_t nmix, const int32_t* idx, const double* weight, int32_t nrec, const double* E, double* e,
            double* q, int32_t* any) {
  for (int32_t c = 0; c < ncol; c++) {
    bool a = false;
    q[c] = 0.0;
    for (int m = 0; m < nmix; m++)
      if (idx[c * nmix + m] >= 0) noise_accumulate(q[c], a, weight[c * nmix + m], weight[c * nmix + m]);
    any[c] = a;
    for (int32_t r = 0; r < nrec; r++) {
      double x = 0.0;
      bool got = false;
      for (int m = 0; m < nmix; m++) {
        const int32_t b = idx[c * nmix + m];
        if (b >= 0) noise_accumulate(x, got, weight[c * nmix + m], E[(int64_t)b * nrec + r]);
      }
      e[(int64_t)c * nrec + r] = x;
    }
  }
}

// out[j] = v[j] perturbed by the mixed e[j] of a column with sum of squared weights q[j]
void nh_apply_mixed(int32_t mode, double sigma, int64_t n, const double* v, const double* e, const double* q, double* out) {
  const NoiseKind nk = noise_kind(sigma, 0.5, mode);
  for (int64_t j = 0; j < n; j++) out[j] = noise_apply_mixed(nk, v[j], e[j], q[j]);
}

}  // extern "C"
