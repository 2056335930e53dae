// group_stats.cuh -- ensemble statistics per column group at every S8 record (samsim_b200_set_group_stats).
//
// The rules that fix every bit of the result live here as plain functions, so that tests/hostbuild can compile them
// for the host: the padded member layout (which makes the chunked GPU tree equal the whole pairwise tree), the regrid
// of a snapshot onto the depth grid, the combination of two partial trees and the final count/mean/variance.  The
// kernels that use them are in samsim_b200.cu.
//
// The tree.  The members of a group, in ascending caller column order, are padded with +0.0 to the next power of two
// P, and the sum is a = a[0::2] + a[1::2] repeated.  Each group occupies P consecutive entries of the padded member
// array, and groups are placed by P descending, so every group starts at a multiple of its own P (and of the tile
// size when P exceeds it).  A tile of 1,024 entries then holds either whole groups or one aligned chunk of one group;
// an xor butterfly over the lanes of a tile adds exactly the adjacent pairs of the tree (IEEE addition commutes), and
// the same tree over the chunk sums of a large group completes it.
#pragma once

#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <vector>

#define SAMSIM_GS_TILE 1024  // entries (threads) of one tile of the reduction kernels
#define SAMSIM_GS_NSC 20     // the SAMSIM_SNAPSC_* scalars, quantities 0..19

namespace samsim {

// Padded member layout of one group assignment (host).  entry t of the padded array holds caller column col[t] (-1:
// padding), and info[t] = group << 5 | log2(P) of the group it belongs to (-1: tail padding past the last group).
// Empty groups get one padding entry (P = 1), so they are reduced like the others and come out with count 0.
struct GsLayout {
  std::vector<int32_t> col, info;
  std::vector<int64_t> start;  // [ngroup] first entry of each group
  std::vector<int32_t> lg;     // [ngroup] log2(P)
  int64_t npad = 0;            // multiple of SAMSIM_GS_TILE
};

__host__ __device__ inline int gs_log2_ceil(int64_t n) {
  int l = 0;
  while ((int64_t(1) << l) < n) l++;
  return l;
}

// group_of_col: [ncol] in [-1, ngroup), nullptr = every column in group 0
inline GsLayout gs_layout(int64_t ncol, int32_t ngroup, const int32_t* group_of_col) {
  GsLayout L;
  std::vector<int64_t> n((size_t)ngroup, 0);
  for (int64_t c = 0; c < ncol; c++) {
    const int g = group_of_col ? group_of_col[c] : 0;
    if (g >= 0) n[(size_t)g]++;
  }
  L.lg.resize((size_t)ngroup);
  std::vector<int32_t> order((size_t)ngroup);
  for (int32_t g = 0; g < ngroup; g++) {
    L.lg[(size_t)g] = gs_log2_ceil(std::max<int64_t>(n[(size_t)g], 1));
    order[(size_t)g] = g;
  }
  std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return L.lg[(size_t)a] > L.lg[(size_t)b]; });
  L.start.resize((size_t)ngroup);
  int64_t off = 0;
  for (int32_t g : order) {
    L.start[(size_t)g] = off;
    off += int64_t(1) << L.lg[(size_t)g];
  }
  L.npad = (off + SAMSIM_GS_TILE - 1) / SAMSIM_GS_TILE * SAMSIM_GS_TILE;
  L.col.assign((size_t)L.npad, -1);
  L.info.assign((size_t)L.npad, -1);
  for (int32_t g = 0; g < ngroup; g++)
    for (int64_t k = 0; k < (int64_t(1) << L.lg[(size_t)g]); k++) L.info[(size_t)(L.start[(size_t)g] + k)] = (g << 5) | L.lg[(size_t)g];
  std::vector<int64_t> fill(L.start);
  for (int64_t c = 0; c < ncol; c++) {
    const int g = group_of_col ? group_of_col[c] : 0;
    if (g >= 0) L.col[(size_t)(fill[(size_t)g]++)] = (int32_t)c;
  }
  return L;
}

// Regrid of one snapshot column onto the depths z[0..nz) (sorted, > 0): D_k = (((thick(1) + thick(2)) + ...) +
// thick(k)); depth j takes layer k, the smallest k <= n_active with z[j] <= D_k.  Calls emit(j, k) for every depth
// that is reached and returns D_{n_active}; depths below it are not reached (the member does not contribute there).
template <class Thick, class Emit>
__host__ __device__ inline double gs_regrid(const Thick& thick, int n_active, const double* z, int nz, Emit emit) {
  double D = 0.0;
  int j = 0;
  for (int k = 1; k <= n_active; k++) {
    D = D + thick(k);
    for (; j < nz && z[j] <= D; j++) emit(j, k);
  }
  return D;
}

// A partial tree: sum, contributing count, min, max (NaN = no contributor, which fmin / fmax skip)
struct GsAcc {
  double s, n, mn, mx;
};
__host__ __device__ inline GsAcc gs_combine(const GsAcc& a, const GsAcc& b) {
  return GsAcc{a.s + b.s, a.n + b.n, fmin(a.mn, b.mn), fmax(a.mx, b.mx)};
}
// statistics of a group from its count and the two tree sums: mean = S / count, variance = M2 / (count - 1)
__host__ __device__ inline double gs_mean(double n, double s) { return (n > 0.0) ? s / n : nan(""); }
__host__ __device__ inline double gs_variance(double n, double m2) {
  return (n >= 2.0) ? m2 / (n - 1.0) : (n == 1.0) ? 0.0 : nan("");
}

}  // namespace samsim
