// noise.cuh -- stochastic forcing perturbations (samsim_b200_set_stochastic_forcing): per-column AR(1) red noise on the
// records of the reanalysis forcing, generated where it is used from a counter-based generator.
//
// The rules that fix every bit live here as plain functions, so that tests/hostbuild can compile them for the host:
// the generator, the normal deviate, the recursion, the three modes and the cursor rule of the window kernel.  The
// kernels that use them are in samsim_b200.cu.
//
// Contract.  Per forcing kind k (samsim_forcing_kind order) the batch has sigma[k] >= 0, phi[k] in [0, 1) and a mode.
// For stream s >= 0, kind k and table record r >= 1 (1-based, the record numbering of samsim_b200_set_forcing):
//   (x0,x1,x2,x3) = Philox4x32-10(counter = (r, k, s, 0), key = (seed & 0xffffffff, seed >> 32))   (Random123)
//   u1 = ((double)(x0 >> 6) * 2^26 + (double)(x1 >> 6) + 0.5) * 2^-52        in (0, 1), exact
//   u2 = ((double)(x2 >> 6) * 2^26 + (double)(x3 >> 6) + 0.5) * 2^-52
//   z(r) = sqrt(-2.0 * det_log(u1)) * det_cos(6.283185307179586 * u2)
//   e(1) = sigma * z(1)                                   stationary from the first record
//   e(r) = phi * e(r-1) + c * z(r),   c = sigma * sqrt(1.0 - phi * phi)
// every operation rounded on its own (-fmad=false on the device, -ffp-contract=off on the host).  The record value
// v = base * scale + offset becomes
//   mode 0, additive:        v + e
//   mode 1, multiplicative:  v * fmax(1.0 + e, 0.0)
//   mode 2, lognormal:       v * det_exp(e - h),  h = 0.5 * (sigma * sigma)   (the mean of v is kept)
// A kind with sigma 0 and a column with stream -1 read v unchanged.  The noise is keyed on the table record, not on
// the step or the launch, so it does not depend on launch lengths, re-binning, shards or restarts.
//
// Correlated noise (samsim_b200_set_stochastic_forcing_correlated, DESIGN §7.4) generalises this.  A column mixes up to
// SAMSIM_NOISE_MAXMIX basis streams, and the kinds' innovations are correlated through a 4x4 matrix corr.  For basis
// stream b >= 0 and record r, z_k(r; b) is z(r) above with s = b, drawn for all four kinds whatever their sigma, and
//   w_k = z_k                                                   corr NULL or the identity: no arithmetic
//   w_k = ((L[k][0]*z_0 + L[k][1]*z_1) + ...) + L[k][k]*z_k     otherwise, left to right
// with L the Cholesky factor of corr (noise_cholesky, in double, at set time).  E_k(1) = sigma_k * w_k(1) and
// E_k(r) = phi_k * E_k(r-1) + c_k * w_k(r).  Column c holds entries m = 0..nmix-1, a basis id (-1 = empty) and a
// finite weight; over its non-empty entries in m order
//   e = w * E(b) of the first, then e = e + w * E(b)        (from the first term, not from 0.0: -0.0 is kept)
//   q = w * w of the first, then q = q + w * w
// and the modes read e, with h * q in place of h for the lognormal one.  A column with no entry reads v unchanged.
// One entry of weight 1.0 with corr the identity gives the bits of the single-stream contract above.
#pragma once

#include <math.h>
#include <stdint.h>

#include "detmath.h"

#define SAMSIM_NOISE_ADDITIVE 0
#define SAMSIM_NOISE_MULTIPLICATIVE 1
#define SAMSIM_NOISE_LOGNORMAL 2
#define SAMSIM_NOISE_MAXMIX 8

namespace samsim {

// the batch-wide setting of one kind; c and h are derived by noise_kind
struct NoiseKind {
  double sigma, phi, c, h;
  int mode;
};

__host__ __device__ inline NoiseKind noise_kind(double sigma, double phi, int mode) {
  NoiseKind k;
  k.sigma = sigma;
  k.phi = phi;
  k.c = sigma * sqrt(1.0 - phi * phi);
  k.h = 0.5 * (sigma * sigma);
  k.mode = mode;
  return k;
}

// Philox4x32 with 10 rounds (Salmon et al. 2011, Random123), in place on the counter
__host__ __device__ inline void philox4x32_10(uint32_t x[4], uint32_t k0, uint32_t k1) {
  for (int round = 0; round < 10; round++) {
    if (round > 0) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    const uint64_t p0 = (uint64_t)0xD2511F53u * x[0];
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * x[2];
    const uint32_t y0 = (uint32_t)(p1 >> 32) ^ x[1] ^ k0;
    const uint32_t y2 = (uint32_t)(p0 >> 32) ^ x[3] ^ k1;
    x[0] = y0;
    x[1] = (uint32_t)p1;
    x[2] = y2;
    x[3] = (uint32_t)p0;
  }
}

// 52 random bits of two words, centred in their interval: in (0, 1), no rounding
__host__ __device__ inline double noise_uniform(uint32_t a, uint32_t b) {
  return ((double)(a >> 6) * 67108864.0 + (double)(b >> 6) + 0.5) * (1.0 / 4503599627370496.0);
}

// z(r) of stream s >= 0 and kind k (Box-Muller on one Philox block)
__host__ __device__ inline double noise_normal(uint64_t seed, int kind, int32_t stream, int32_t rec) {
  uint32_t x[4] = {(uint32_t)rec, (uint32_t)kind, (uint32_t)stream, 0u};
  philox4x32_10(x, (uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32));
  const double u1 = noise_uniform(x[0], x[1]), u2 = noise_uniform(x[2], x[3]);
  return sqrt(-2.0 * det_log(u1)) * det_cos(6.283185307179586 * u2);
}

// e(rec) from e(rec-1) (ignored for rec 1)
__host__ __device__ inline double noise_next(const NoiseKind& nk, double e_prev, double z, int32_t rec) {
  return (rec == 1) ? nk.sigma * z : nk.phi * e_prev + nk.c * z;
}

// the record value v perturbed by e
__host__ __device__ inline double noise_apply(const NoiseKind& nk, double v, double e) {
  if (nk.mode == SAMSIM_NOISE_ADDITIVE) return v + e;
  if (nk.mode == SAMSIM_NOISE_MULTIPLICATIVE) return v * fmax(1.0 + e, 0.0);
  return v * det_exp(e - nk.h);
}

// Cursor rule.  The device keeps e(cursor-1) and e(cursor) of every column and kind; cursor is batch-wide and 0 while
// nothing is held.  A window of records first..last that starts at cursor-1 or later advances from the held values,
// an earlier one (set_clock moved back, a checkpoint loaded, a new setting) restarts from record 1.  Either way e(r) is
// the same pure function of the record.
__host__ __device__ inline bool noise_resumes(int32_t cursor, int32_t first) { return cursor >= 1 && first >= cursor - 1; }
__host__ __device__ inline int32_t noise_cursor_after(int32_t cursor, int32_t first, int32_t last) {
  return (noise_resumes(cursor, first) && cursor > last) ? cursor : last;
}

// e(r) of one stream and kind for r = first..last, passed to emit(r, e) in record order; ep, ec hold e(cursor-1) and
// e(cursor) on entry and e(c'-1), e(c') on return, c' = noise_cursor_after(cursor, first, last)
template <class Emit>
__host__ __device__ inline void noise_window(const NoiseKind& nk, uint64_t seed, int kind, int32_t stream, int32_t cursor,
                                             int32_t first, int32_t last, double& ep, double& ec, Emit emit) {
  int32_t at = cursor;  // ep = e(at-1), ec = e(at)
  if (!noise_resumes(cursor, first)) {
    at = 0;
    ep = ec = 0.0;
  }
  for (int32_t r = first; r <= last; r++) {
    while (at < r) {
      at++;
      ep = ec;
      ec = noise_next(nk, ec, noise_normal(seed, kind, stream, at), at);
    }
    emit(r, (r == at) ? ec : ep);
  }
}

// ---- correlated noise --------------------------------------------------------------------------------------------

// The Cholesky factor of the kinds' correlation: on == 0 for the identity (w = z, no arithmetic), else L row-major
struct NoiseCorr {
  double L[16];
  int on;
};

// Cholesky-Banachiewicz of the symmetric 4x4 corr (row-major) into L, zero above the diagonal, each operation rounded
// on its own.  False when a pivot is not > 0 (corr not positive definite, or not finite).
__host__ __device__ inline bool noise_cholesky(const double corr[16], double L[16]) {
  for (int q = 0; q < 16; q++) L[q] = 0.0;
  for (int i = 0; i < 4; i++)
    for (int j = 0; j <= i; j++) {
      double s = corr[i * 4 + j];
      for (int m = 0; m < j; m++) s = s - L[i * 4 + m] * L[j * 4 + m];
      if (i == j) {
        if (!(s > 0.0)) return false;
        L[i * 4 + i] = sqrt(s);
      } else {
        L[i * 4 + j] = s / L[j * 4 + j];
      }
    }
  return true;
}

// the four kinds' innovations w of basis stream b at record rec
__host__ __device__ inline void noise_innovations(const NoiseCorr& nc, uint64_t seed, int32_t b, int32_t rec, double w[4]) {
  double z[4];
#pragma unroll
  for (int k = 0; k < 4; k++) z[k] = noise_normal(seed, k, b, rec);
#pragma unroll
  for (int k = 0; k < 4; k++) {
    if (!nc.on) {
      w[k] = z[k];
      continue;
    }
    double s = nc.L[k * 4] * z[0];
#pragma unroll
    for (int j = 1; j <= k; j++) s = s + nc.L[k * 4 + j] * z[j];
    w[k] = s;
  }
}

// noise_window for the four kinds of basis stream b at once: E_k(r) for r = first..last passed to emit(r, E) in record
// order; ep[k], ec[k] hold E_k(cursor-1), E_k(cursor) on entry and on return, under the same cursor rule
template <class Emit>
__host__ __device__ inline void noise_basis_window(const NoiseKind* nk, const NoiseCorr& nc, uint64_t seed, int32_t b,
                                                   int32_t cursor, int32_t first, int32_t last, double ep[4],
                                                   double ec[4], Emit emit) {
  int32_t at = cursor;  // ep = E(at-1), ec = E(at)
  if (!noise_resumes(cursor, first)) {
    at = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) ep[k] = ec[k] = 0.0;
  }
  for (int32_t r = first; r <= last; r++) {
    while (at < r) {
      at++;
      double w[4];
      noise_innovations(nc, seed, b, at, w);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        ep[k] = ec[k];
        ec[k] = noise_next(nk[k], ec[k], w[k], at);
      }
    }
    double E[4];
#pragma unroll
    for (int k = 0; k < 4; k++) E[k] = (r == at) ? ec[k] : ep[k];
    emit(r, E);
  }
}

// One term of a column's mix, in m order over its non-empty entries: acc = w * x for the first (any false on entry),
// acc = acc + w * x after.  x = E(b) gives e, x = w gives q.
__host__ __device__ inline void noise_accumulate(double& acc, bool& any, double w, double x) {
  const double t = w * x;
  acc = any ? acc + t : t;
  any = true;
}

// the record value v perturbed by the column's mixed e, q its sum of squared weights (lognormal: h * q in place of h)
__host__ __device__ inline double noise_apply_mixed(const NoiseKind& nk, double v, double e, double q) {
  if (nk.mode == SAMSIM_NOISE_LOGNORMAL) return v * det_exp(e - nk.h * q);
  return noise_apply(nk, v, e);
}

// The argument rules of both setters, on the host: nullptr for a valid setting, else what is wrong.  basis[c*nmix + m]
// (nullptr = stream c, nmix 1), weight likewise (nullptr = 1.0), corr row-major (nullptr = the identity).  On success
// `on` tells whether a sigma is > 0, `single` whether the setting is the single-stream case (nmix 1, every weight 1.0,
// corr the identity) and nc holds the Cholesky factor (nc.on = 0 for the identity).
inline const char* noise_check(const double sigma[4], const double phi[4], const int32_t mode[4], const double* corr,
                               int32_t nmix, int64_t ncol, const int32_t* basis, const double* weight, bool& on,
                               bool& single, NoiseCorr& nc) {
  on = false;
  for (int k = 0; k < 4; k++) {
    if (!(sigma[k] >= 0.0 && isfinite(sigma[k]))) return "sigma must be finite and >= 0";
    if (!(phi[k] >= 0.0 && phi[k] < 1.0)) return "phi must lie in [0, 1)";
    if (mode[k] < SAMSIM_NOISE_ADDITIVE || mode[k] > SAMSIM_NOISE_LOGNORMAL)
      return "mode must be 0 (additive), 1 (multiplicative) or 2 (lognormal)";
    on = on || sigma[k] > 0.0;
  }
  if (nmix < 1 || nmix > SAMSIM_NOISE_MAXMIX) return "nmix must lie in 1..8";
  if (basis)
    for (int64_t c = 0; c < ncol; c++)
      for (int m = 0; m < nmix; m++) {
        const int32_t b = basis[c * nmix + m];
        if (b < -1) return "stream ids must be >= -1";
        for (int m2 = 0; m2 < m && b >= 0; m2++)
          if (basis[c * nmix + m2] == b) return "basis ids must be distinct within a column";
      }
  bool unit = true;
  if (weight)
    for (int64_t q = 0; q < ncol * nmix; q++) {
      if (!isfinite(weight[q])) return "weights must be finite";
      unit = unit && weight[q] == 1.0;
    }
  for (int q = 0; q < 16; q++) nc.L[q] = 0.0;
  nc.on = 0;
  if (corr) {
    for (int i = 0; i < 4; i++)
      for (int j = 0; j < 4; j++) {
        const double x = corr[i * 4 + j];
        if (!isfinite(x) || x != corr[j * 4 + i] || (i == j && x != 1.0))
          return "corr must be finite, exactly symmetric and have a unit diagonal";
        nc.on = nc.on || (i != j && x != 0.0);
      }
    if (!noise_cholesky(corr, nc.L)) return "corr must be positive definite";
  }
  single = nmix == 1 && unit && !nc.on;
  return nullptr;
}

}  // namespace samsim
