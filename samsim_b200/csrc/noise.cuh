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
#pragma once

#include <math.h>
#include <stdint.h>

#include "detmath.h"

#define SAMSIM_NOISE_ADDITIVE 0
#define SAMSIM_NOISE_MULTIPLICATIVE 1
#define SAMSIM_NOISE_LOGNORMAL 2

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

}  // namespace samsim
