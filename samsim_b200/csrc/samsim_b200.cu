// samsim_b200.cu -- step kernel and the C ABI of include/samsim_b200.h.
//
// Build (see __graft_entry__.build): nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo
// There is no CPU fallback: without a CUDA device samsim_b200_create returns SAMSIM_ERR_NO_DEVICE.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "../../include/samsim_b200.h"
#include "group_stats.cuh"
#include "step.cuh"
#include "time_stats.cuh"

using namespace samsim;

static_assert((int)SAMSIM_SC_COUNT == (int)SC_COUNT, "scalar ids out of sync with include/samsim_b200.h");
static_assert((int)SAMSIM_ARR_COUNT == (int)AR_STATE_COUNT + 2 && (int)SAMSIM_ARR_BGC_ABS1 == (int)AR_STATE_COUNT,
              "array ids out of sync with include/samsim_b200.h");
static_assert((int)SAMSIM_INT_COUNT == (int)IN_COUNT, "int ids out of sync with include/samsim_b200.h");
static_assert((int)SAMSIM_EV_COUNT == (int)EV_COUNT && (int)SAMSIM_EV_TWO_PASS_STEP == (int)EV_TWO_PASS_STEP && (int)SAMSIM_EV_GAS_REFILL == 32,
              "event ids out of sync with include/samsim_b200.h");
static_assert((int)SAMSIM_SNAPSC_COUNT == 20 && (int)SAMSIM_SNAPARR_COUNT == 14, "snapshot layout");

// Launch shape (measured on B200, profiles/README.md): 512-thread blocks, 2 blocks per SM (64 registers/thread,
// 32 warps/SM) and a barrier between the phases of a step (SAMSIM_SYNC, step.cuh).
#ifndef SAMSIM_BLOCK
#define SAMSIM_BLOCK 512
#endif
#ifndef SAMSIM_MINBLOCKS
#define SAMSIM_MINBLOCKS 2
#endif
#define SAMSIM_MAXWIN 24   // forcing records staged per launch (3-hourly): 22 * 10800 s of model time per launch
// Tables of up to SAMSIM_MAXSITE sites are staged in shared memory per launch; larger ones are read in place from
// global memory (samsim_b200_set_forcing)
#ifndef SAMSIM_MAXSITE
#define SAMSIM_MAXSITE 16
#endif

// ------------------------------------------------------------------------------------------
// kernel parameters
// ------------------------------------------------------------------------------------------
struct KParams {
  double* arr;   // [ncol_pad/32][LS][n_arr][32], see physics.cuh
  int n_arr;
  double* sc;    // [SC_COUNT][ncol_pad]
  int* in;       // [IN_COUNT][ncol_pad]
  long long ncol, ncol_pad;
  int LS;
  // clock at launch
  double time;
  long long i;
  int n_time_out, time_counter;
  int nsteps;
  // forcing
  const double* series;   // [nsite][4][nrec] global; staged when nsite <= SAMSIM_MAXSITE
  int nsite, nrec, win_first, win_len;
  const int* site_of_col; // [ncol_pad] or nullptr
  const double* fscale;   // [4][ncol_pad] or nullptr
  const double* foffset;  // [4][ncol_pad] or nullptr
  const double* lab;      // [nset][4][lab_nrec]
  long long lab_nrec;
  const int* set_of_col;
  // last loop index each column runs (samsim_b200_set_end_step), [ncol_pad] in slot order; nullptr = no column ends
  const int64_t* end_of_col;
  // snapshot
  double* snap_sc;
  double* snap_arr;
  // divergence counters (see the end of samsim_step_kernel): [0] idle lane-layers, [1] all lane-layers, [2] warps whose
  // lanes disagree on the snow class or the status, [3] warps
  unsigned long long* divergence;
};

// status of a column that has passed its end step, inside the step kernel only (padding columns hold -1, failed
// ones the reference's positive STOP code); never written back
#define STATUS_FINISHED (-2)

__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem_src));
}

template <bool TWO_PASS>
__global__ void __launch_bounds__(SAMSIM_BLOCK, SAMSIM_MINBLOCKS) samsim_step_kernel(const __grid_constant__ KParams p) {
  __shared__ double s_win[SAMSIM_MAXSITE * 4 * SAMSIM_MAXWIN];
  const bool staged = (p.nsite <= SAMSIM_MAXSITE);
  // stage the forcing window: records win_first .. win_first+win_len-1 of every site/kind (cp.async)
  if (p.series != nullptr && staged) {
    const int n = p.nsite * 4 * p.win_len;
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const int sk = e / p.win_len, r = e - sk * p.win_len;
      cp_async8(&s_win[e], p.series + (size_t)sk * p.nrec + (p.win_first - 1 + r));
    }
    asm volatile("cp.async.commit_group;\n" ::);
    asm volatile("cp.async.wait_group 0;\n" ::);
  }
  __syncthreads();

  // Padding threads (col >= ncol, same block) stay in the loop for the phase barriers with status = -1; the
  // buffers are allocated to ncol_pad so their loads are in bounds.
  const long long col_raw = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool padding = (col_raw >= p.ncol);
  const long long col = padding ? (p.ncol - 1) : col_raw;
  const size_t ls = (size_t)p.ncol_pad;  // row stride of the scalar / int / forcing rows

  Col c;
  c.ls = (unsigned)(p.n_arr * SAMSIM_TILE);
  c.base = p.arr + (size_t)(col / SAMSIM_TILE) * p.LS * c.ls + (size_t)(col % SAMSIM_TILE);
  for (int q = 0; q < SC_COUNT; q++) c.sc[q] = p.sc[(size_t)q * ls + col];
  c.N_active = p.in[(size_t)IN_N_ACTIVE * ls + col];
  c.status = padding ? -1 : p.in[(size_t)IN_STATUS * ls + col];
  c.styropor_flag = p.in[(size_t)IN_STYROPOR * ls + col];
  c.ev0 = (unsigned)p.in[(size_t)IN_EVENTS0 * ls + col];
  c.ev1 = (unsigned)p.in[(size_t)IN_EVENTS1 * ls + col];
  c.time = p.time; c.i = p.i; c.n_time_out = p.n_time_out; c.time_counter = p.time_counter;
  c.fsw0 = c.fsw1 = c.flw0 = c.flw1 = c.ftime0 = c.ftime1 = 0.0;
  c.thermo_valid = false;  // launch-local: the host may have changed the state between launches
  c.pre.valid = false;
  c.want_state = false;
  c.fb.tot_valid = c.fb.suf_valid = c.fb.res_valid = false; c.fb.k_last = 0; c.fb.ks = 0;
  c.min_psi_s = 0.0; c.min_S_abs_2 = 0.0;
  c.fb_x = 0.0;

  Forcing f;
  if (staged) {
    f.win = s_win; f.win_len = p.win_len; f.win_first = p.win_first;
  } else {  // the table as samsim_b200_set_forcing stored it
    f.win = p.series; f.win_len = p.nrec; f.win_first = 1; f.global = true;
  }
  f.site = p.site_of_col ? p.site_of_col[col] : 0;
  for (int k = 0; k < 4; k++) {
    f.scale[k] = p.fscale ? p.fscale[(size_t)k * ls + col] : 1.0;
    f.offset[k] = p.foffset ? p.foffset[(size_t)k * ls + col] : 0.0;
  }
  f.lab = p.lab; f.lab_nrec = p.lab_nrec;
  f.lab_set = p.set_of_col ? p.set_of_col[col] : 0;

  SnapOut snap;
  snap.scalars = p.snap_sc; snap.arrays = p.snap_arr; snap.ncol_pad = ls; snap.col = (int)col;

  // A column runs loop index i only while i <= its end step.  From then on it is frozen like a failed column: its
  // status holds STATUS_FINISHED for the rest of the launch and 0 again on write-back.
  int my_steps = p.nsteps;
  if (p.end_of_col) {
    const long long left = p.end_of_col[col] - p.i;
    my_steps = (left <= 0) ? 0 : (left < p.nsteps) ? (int)left : p.nsteps;
  }
  // every thread runs every step: a failed or finished column only skips the phase bodies (column_step checks
  // c.status).  A column's last step materialises what a launch otherwise only writes at its end (S_bu, ray, fl_Q, the
  // S0 diagnostics); want_diag at any step leaves the results unchanged, as launches of arbitrary lengths show.
  for (int s = 0; s < p.nsteps; s++) {
    if (s == my_steps && c.status == 0) c.status = STATUS_FINISHED;
    column_step<TWO_PASS>(c, f, s == p.nsteps - 1 || s == my_steps - 1, snap);
  }

  // ---- lane divergence of this launch's end state, measured where it arises: in the warp --------------------------
  // A warp runs every layer sweep to the deepest of its 32 columns and every branch that one of its lanes takes.
  // idle lane-layers = SUM over lanes (max N_active in the warp - N_active of the lane); lanes that disagree on the
  // snow class (the S2 / S3 / S10 / S17 branches), on a melting surface (S20-S21 flushing and the full S4 sweep that
  // follows it) or on being failed are counted per warp with a ballot.  The host
  // re-bins the columns when the idle share crosses its threshold (samsim_b200_set_rebin_auto) instead of on a
  // fixed interval.
  if (p.divergence) {
    const unsigned full = 0xffffffffu;
    const bool live = !padding && c.status == 0;
    const int na = live ? c.N_active : 0;
    const int mx = __reduce_max_sync(full, na);
    const int idle = __reduce_add_sync(full, live ? (mx - na) : 0);
    const int nlive = __popc(__ballot_sync(full, live));
    const double ts = c.sc[SC_THICK_SNOW];
    // + 4 for columns whose surface melted in the last step: they flush (S21) and re-solve every layer in the next S4,
    // and one such lane makes its warp pay for both
    const int cls = !live ? -1 : (((ts <= 0.0) ? 0 : (ts < CFG.thick_min / 100.0) ? 1 : (ts < CFG.thick_min) ? 2 : 3) |
                                  ((c.sc[SC_MELT_THICK] > 0.0) ? 4 : 0));
    const int cls0 = __shfl_sync(full, cls, __ffs(__ballot_sync(full, live)) - 1);
    const unsigned differ = __ballot_sync(full, live && cls != cls0);
    if ((threadIdx.x & 31) == 0 && nlive > 0) {
      atomicAdd(&p.divergence[0], (unsigned long long)idle);
      atomicAdd(&p.divergence[1], (unsigned long long)mx * (unsigned long long)nlive);
      atomicAdd(&p.divergence[2], (unsigned long long)(differ != 0u));
      atomicAdd(&p.divergence[3], 1ull);
    }
  }

  if (padding) return;
  for (int q = 0; q < SC_COUNT; q++) p.sc[(size_t)q * ls + col] = c.sc[q];
  p.in[(size_t)IN_N_ACTIVE * ls + col] = c.N_active;
  p.in[(size_t)IN_STATUS * ls + col] = (c.status == STATUS_FINISHED) ? 0 : c.status;
  p.in[(size_t)IN_STYROPOR * ls + col] = c.styropor_flag;
  p.in[(size_t)IN_EVENTS0 * ls + col] = (int)c.ev0;
  p.in[(size_t)IN_EVENTS1 * ls + col] = (int)c.ev1;
}

// Column -> slot indirection.  After samsim_b200_rebin the columns of a handle sit in regime order; `map`
// (slot_of_col, nullptr = identity) translates the caller's column index in every host-facing kernel.
__device__ __forceinline__ long long slot_of(const int* map, long long col) { return map ? (long long)map[col] : col; }

// element (array slot a, layer k) of the column in device slot s of the tiled state buffer (physics.cuh)
__host__ __device__ __forceinline__ size_t state_index(long long s, int k, int a, int LS, int n_arr) {
  return ((((size_t)(s / SAMSIM_TILE)) * LS + k) * n_arr + a) * SAMSIM_TILE + (size_t)(s % SAMSIM_TILE);
}

// replicate one column (ensemble initialisation)
__global__ void samsim_broadcast_kernel(double* arr, double* sc, int* in, long long ncol_pad, int LS, int src, int col0,
                                        int n, const int* map, int n_arr) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const long long col = slot_of(map, col0 + t);
  src = (int)slot_of(map, src);
  if (col == src) return;
  const size_t ls = (size_t)ncol_pad;
  for (int k = 0; k < LS; k++)
    for (int a = 0; a < n_arr; a++) arr[state_index(col, k, a, LS, n_arr)] = arr[state_index(src, k, a, LS, n_arr)];
  for (int q = 0; q < SC_COUNT; q++) sc[(size_t)q * ls + col] = sc[(size_t)q * ls + src];
  for (int q = 0; q < IN_COUNT; q++) in[(size_t)q * ls + col] = in[(size_t)q * ls + src];
}

// gather a snapshot block into host order: dst[(c*count + id)*ext + (k-1)]
__global__ void samsim_gather_kernel(const double* src, double* dst, long long ncol_pad, int LS, int count, int ext,
                                     int col0, int n, int k0, const int* map) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)n * count * ext;
  if (t >= total) return;
  // t enumerates (id, k, c) with c fastest so reads are coalesced
  const int cc = (int)(t % n);
  const long long r = t / n;
  const int k = (int)(r % ext);
  const int id = (int)(r / ext);
  dst[((size_t)cc * count + id) * ext + k] = src[((size_t)id * LS + (k + k0)) * (size_t)ncol_pad + slot_of(map, col0 + cc)];
}
// state arrays (tiled layout) <-> host order host[c*ext + (k-1)]
__global__ void samsim_state_gather_kernel(const double* arr, double* dst, int LS, int n_arr, int a, int ext, int col0, int n,
                                           const int* map) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * ext) return;
  const int cc = (int)(t % n), k = (int)(t / n);  // column fastest: coalesced reads within a tile row
  dst[(size_t)cc * ext + k] = arr[state_index(slot_of(map, col0 + cc), k + 1, a, LS, n_arr)];
}
__global__ void samsim_scatter_kernel(double* arr, const double* srchost, int LS, int n_arr, int a, int ext, int col0, int n,
                                      const int* map) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)n * ext;
  if (t >= total) return;
  const int cc = (int)(t % n);
  const int k = (int)(t / n);
  arr[state_index(slot_of(map, col0 + cc), k + 1, a, LS, n_arr)] = srchost[(size_t)cc * ext + k];
}
// re-binning of one state array: rows[k][s] (k = 0..LS-1, row stride ncol_pad) <-> the tiled buffer
__global__ void samsim_state_to_rows_kernel(const double* arr, double* rows, long long ncol, long long ncol_pad, int LS, int n_arr,
                                            int a, const int* order) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)LS * ncol) return;
  const long long k = t / ncol, s = t - k * ncol;
  rows[k * ncol_pad + s] = arr[state_index(order[s], (int)k, a, LS, n_arr)];
}
__global__ void samsim_rows_to_state_kernel(double* arr, const double* rows, long long ncol, long long ncol_pad, int LS, int n_arr, int a) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)LS * ncol) return;
  const long long k = t / ncol, s = t - k * ncol;
  arr[state_index(s, (int)k, a, LS, n_arr)] = rows[k * ncol_pad + s];
}
// per-column vectors (scalars, ints, forcing perturbations) through the slot map
template <typename T>
__global__ void samsim_vec_get_kernel(const T* row, T* dst, int col0, int n, const int* map) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) dst[t] = row[slot_of(map, col0 + t)];
}
template <typename T>
__global__ void samsim_vec_set_kernel(T* row, const T* src, int col0, int n, const int* map) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) row[slot_of(map, col0 + t)] = src[t];
}

// ---- re-binning (SURVEY 8e: columns are re-binned by regime for warp coherence; local permutation only) ----
// key: failed and finished columns last; then N_active descending (loop trip counts), snow class (the snow branches) and melting
// surface (flushing, full S4 sweep), forcing site, surface temperature.  Bits from the top: idle (1), 0xFFF - N_active (12),
// class (3), site (site_bits, the whole site index), T_top bucket (10).
__global__ void samsim_rebin_key_kernel(const double* sc, const int* in, const int* site_of_col, const int64_t* end_of_col,
                                        long long i, long long ncol, long long ncol_pad, double thick_min, int site_bits,
                                        unsigned long long* keys, int* vals) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= ncol) return;
  const int na = in[(size_t)IN_N_ACTIVE * ncol_pad + s];
  // a finished column idles like a failed one: their warps should hold no running column
  const bool idle = in[(size_t)IN_STATUS * ncol_pad + s] != 0 || (end_of_col && end_of_col[s] <= i);
  const double snow = sc[(size_t)SC_THICK_SNOW * ncol_pad + s];
  const unsigned cls = ((snow <= 0.0) ? 0u : (snow < thick_min / 100.0) ? 1u : (snow < thick_min) ? 2u : 3u) |
                       ((sc[(size_t)SC_MELT_THICK * ncol_pad + s] > 0.0) ? 4u : 0u);  // melting surface: the flushing / full-S4 path
  const unsigned long long site = site_of_col ? (unsigned)site_of_col[s] : 0u;
  // deepest columns first: blocks are dispatched in index order, so the cheap ones fill the tail of the launch
  // within a site, columns with a similar surface temperature (0.1 K buckets over -80..+22 degC) sit next to each other:
  // their Newton sweeps take the same number of iterations and their drainage candidates span the same layers
  const double tt = sc[(size_t)SC_T_TOP * ncol_pad + s];
  const unsigned tb = (tt > -80.0) ? ((tt < 22.3) ? (unsigned)((tt + 80.0) * 10.0) : 1023u) : 0u;  // NaN -> 0
  const int b = 10 + site_bits;
  keys[s] = ((idle ? 1ull : 0ull) << (b + 15)) | ((unsigned long long)(0xFFFu - ((unsigned)na & 0xFFFu)) << (b + 3)) |
            ((unsigned long long)cls << b) | (site << 10) | tb;
  vals[s] = (int)s;
}
__global__ void samsim_rebin_unsorted_kernel(const unsigned long long* keys, long long ncol, int* out) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s + 1 < ncol && keys[s] > keys[s + 1]) atomicAdd(out, 1);
}
// tmp[row][s] = src[row][order[s]] for the real columns; padding columns keep their place
template <typename T>
__global__ void samsim_permute_rows_kernel(const T* src, T* tmp, long long ncol, long long ncol_pad, int nrows, const int* order) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)nrows * ncol_pad) return;
  const long long row = t / ncol_pad, s = t - row * ncol_pad;
  tmp[t] = (s < ncol) ? src[row * ncol_pad + order[s]] : src[t];
}
__global__ void samsim_rebin_maps_kernel(const int* order, const int* old_col_of_slot, int* new_col_of_slot, int* slot_of_col, long long ncol) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= ncol) return;
  const int col = old_col_of_slot ? old_col_of_slot[order[s]] : order[s];
  new_col_of_slot[s] = col;
  slot_of_col[col] = (int)s;
}

// block partial reductions for reduce_diag: out[block][6][3]
__global__ void samsim_reduce_kernel(const double* sc, const int* in, long long ncol, long long ncol_pad, double* out) {
  __shared__ double sh[6][3][128];
  const long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int ids[5] = {SC_THICKNESS, SC_BULK_SALIN, SC_FREEBOARD, SC_THICK_SNOW, SC_T_TOP};
  for (int j = 0; j < 6; j++) {
    double v = 0.0, mn = 1e300, mx = -1e300;
    if (col < ncol) {
      v = (j < 5) ? sc[(size_t)ids[j] * ncol_pad + col] : (double)in[(size_t)IN_N_ACTIVE * ncol_pad + col];
      mn = v; mx = v;
    }
    sh[j][0][threadIdx.x] = v; sh[j][1][threadIdx.x] = mn; sh[j][2][threadIdx.x] = mx;
  }
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s)
      for (int j = 0; j < 6; j++) {
        sh[j][0][threadIdx.x] += sh[j][0][threadIdx.x + s];
        sh[j][1][threadIdx.x] = fmin(sh[j][1][threadIdx.x], sh[j][1][threadIdx.x + s]);
        sh[j][2][threadIdx.x] = fmax(sh[j][2][threadIdx.x], sh[j][2][threadIdx.x + s]);
      }
    __syncthreads();
  }
  if (threadIdx.x == 0)
    for (int j = 0; j < 6; j++)
      for (int q = 0; q < 3; q++) out[((size_t)blockIdx.x * 6 + j) * 3 + q] = sh[j][q][0];
}

// ---- group statistics at S8 records (group_stats.cuh; samsim_b200_set_group_stats) --------------------------------
struct GsParams {
  // snapshot, status and end steps, all in slot order
  const double* snap_sc;   // [SNAPSC_COUNT][ncol_pad]
  const double* snap_arr;  // [SNAPARR_COUNT][LS][ncol_pad]
  const int* in;
  const int64_t* end_of_col;
  const int* map;          // slot_of_col, nullptr = identity
  long long ncol_pad;
  int LS;
  long long i;             // loop index of the record
  // padded member layout (GsLayout)
  const int* col;
  const int* info;
  long long npad;
  const double* z;
  int nz, nprof, Q;
  int prof[SAMSIM_SNAPARR_COUNT];  // selected snapshot arrays, ascending
  double* vals;            // [Q][npad]
  double* reach;           // [npad]: -inf = not contributing, else D_{N_active} of the member's snapshot
  double *pS, *pN, *pMn, *pMx;  // [Q][npad / SAMSIM_GS_TILE] chunk sums of groups larger than a tile
  const int* big_group;    // groups larger than a tile
  double* out;             // this record: [ngroup][Q][5] = count, mean, variance, min, max
};

// one thread per padded entry: the member's quantities in [q][entry] order (coalesced writes)
__global__ void samsim_gs_gather_kernel(const GsParams p) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= p.npad) return;
  const int c = p.col[t];
  double reach = -INFINITY;
  if (c >= 0) {
    const long long s = slot_of(p.map, c);
    const size_t ls = (size_t)p.ncol_pad;
    // failed and finished columns hold stale snapshots
    if (p.in[(size_t)IN_STATUS * ls + s] == 0 && (!p.end_of_col || p.end_of_col[s] >= p.i)) {
      const size_t np = (size_t)p.npad;
      for (int q = 0; q < SAMSIM_GS_NSC; q++) p.vals[q * np + t] = p.snap_sc[q * ls + s];
      reach = 0.0;
      if (p.nprof > 0) {
        const double* A = p.snap_arr;
        const int LS = p.LS;
        const int na = (int)p.snap_sc[(size_t)SAMSIM_SNAPSC_N_ACTIVE * ls + s];
        auto thick = [&](int k) { return A[((size_t)SAMSIM_SNAPARR_THICK * LS + k) * ls + s]; };
        reach = gs_regrid(thick, na, p.z, p.nz, [&](int j, int k) {
          for (int a = 0; a < p.nprof; a++)
            p.vals[(size_t)(SAMSIM_GS_NSC + a * p.nz + j) * np + t] = A[((size_t)p.prof[a] * LS + k) * ls + s];
        });
      }
    }
  }
  p.reach[t] = reach;
}

template <bool S_ONLY>
__device__ __forceinline__ GsAcc gs_shfl(const GsAcc& a, int o) {
  const unsigned full = 0xffffffffu;
  GsAcc b;
  b.s = __shfl_xor_sync(full, a.s, o);
  if (S_ONLY) return b;
  b.n = __shfl_xor_sync(full, a.n, o);
  b.mn = __shfl_xor_sync(full, a.mn, o);
  b.mx = __shfl_xor_sync(full, a.mx, o);
  return b;
}
template <bool S_ONLY>
__device__ __forceinline__ GsAcc gs_add(const GsAcc& a, const GsAcc& b) {
  if (S_ONLY) return GsAcc{a.s + b.s, a.n, a.mn, a.mx};
  return gs_combine(a, b);
}

// Pairwise tree over aligned blocks of 2^lgw (<= SAMSIM_GS_TILE) threads: each thread holds one leaf and the lgw of
// its block (uniform over the block).  emit(first thread of the block, g, result) is called once per block.  All
// threads of the block of SAMSIM_GS_TILE must call it.
template <bool S_ONLY, class Emit>
__device__ __forceinline__ void gs_block_tree(GsAcc a, int lgw, int g, Emit emit) {
  __shared__ double sh[4][32];
  __shared__ int shl[32], shg[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    const GsAcc b = gs_shfl<S_ONLY>(a, o);
    if (o < (1 << lgw)) a = gs_add<S_ONLY>(a, b);
  }
  if (lgw <= 5 && (lane & ((1 << lgw) - 1)) == 0) emit((int)threadIdx.x, g, a);
  if (lane == 0) { sh[0][warp] = a.s; sh[1][warp] = a.n; sh[2][warp] = a.mn; sh[3][warp] = a.mx; shl[warp] = lgw; shg[warp] = g; }
  __syncthreads();
  if (warp == 0) {
    GsAcc x{sh[0][lane], sh[1][lane], sh[2][lane], sh[3][lane]};
    const int l2 = shl[lane] - 5;  // levels above the warp
    for (int o = 1; o < 32; o <<= 1) {
      const GsAcc b = gs_shfl<S_ONLY>(x, o);
      if (l2 > 0 && o < (1 << l2)) x = gs_add<S_ONLY>(x, b);
    }
    if (l2 > 0 && (lane & ((1 << l2) - 1)) == 0) emit(lane * 32, shg[lane], x);
  }
  __syncthreads();
}

// One tile of SAMSIM_GS_TILE padded entries per block, every quantity.  Pass 1 (SECOND = false): count, sum, min,
// max; pass 2: the sum of squared deviations from the mean of pass 1.  Groups inside the tile are finished here;
// a group larger than the tile leaves its chunk sum in pS.. for samsim_gs_final_kernel.
template <bool SECOND>
__global__ void __launch_bounds__(SAMSIM_GS_TILE) samsim_gs_tile_kernel(const GsParams p) {
  const long long tile = blockIdx.x, t = tile * SAMSIM_GS_TILE + threadIdx.x;
  const long long ntile = p.npad / SAMSIM_GS_TILE;
  const size_t np = (size_t)p.npad;
  const int info = p.info[t];
  const int g = (info < 0) ? -1 : (info >> 5);
  const int lg = (info < 0) ? 0 : (info & 31);
  const int lgw = (lg < 10) ? lg : 10;
  const double reach = p.reach[t];
  const int Q = p.Q;
  for (int q = 0; q < Q; q++) {
    const double v = p.vals[q * np + t];
    const bool in = (q < SAMSIM_GS_NSC) ? (reach != -INFINITY) : (p.z[(q - SAMSIM_GS_NSC) % p.nz] <= reach);
    GsAcc a;
    if (!SECOND) {
      a = in ? GsAcc{v, 1.0, v, v} : GsAcc{0.0, 0.0, nan(""), nan("")};
    } else {
      const double d = (in && g >= 0) ? v - p.out[((size_t)g * Q + q) * 5 + 1] : 0.0;
      a = GsAcc{d * d, 0.0, 0.0, 0.0};
    }
    gs_block_tree<SECOND>(a, lgw, g, [&](int, int gg, const GsAcc& r) {
      if (gg < 0) return;
      if (lg > 10) {
        const size_t k = (size_t)q * ntile + tile;
        p.pS[k] = r.s;
        if (!SECOND) { p.pN[k] = r.n; p.pMn[k] = r.mn; p.pMx[k] = r.mx; }
        return;
      }
      double* o = p.out + ((size_t)gg * Q + q) * 5;
      if (!SECOND) { o[0] = r.n; o[1] = gs_mean(r.n, r.s); o[3] = r.mn; o[4] = r.mx; }
      else o[2] = gs_variance(o[0], r.s);
    });
  }
}

// Groups larger than a tile: the same tree over their chunk sums, one block per (group, quantity).  Chunk sums are
// reduced in place, SAMSIM_GS_TILE at a time, until one is left.
template <bool SECOND>
__global__ void __launch_bounds__(SAMSIM_GS_TILE) samsim_gs_final_kernel(const GsParams p, const int* start_tile,
                                                                         const int* lg_of) {
  const int b = blockIdx.x, q = blockIdx.y, Q = p.Q;
  const int g = p.big_group[b];
  const long long ntile = p.npad / SAMSIM_GS_TILE;
  const size_t base = (size_t)q * ntile + start_tile[b];
  long long n = 1ll << (lg_of[b] - 10);
  while (n > 1) {
    const int lgw = (n >= SAMSIM_GS_TILE) ? 10 : gs_log2_ceil(n);
    const long long w = 1ll << lgw;
    for (long long c = 0; c < n / w; c++) {
      const size_t k = base + c * w + threadIdx.x;
      GsAcc a{0.0, 0.0, nan(""), nan("")};
      if (threadIdx.x < w) {
        a.s = p.pS[k];
        if (!SECOND) { a.n = p.pN[k]; a.mn = p.pMn[k]; a.mx = p.pMx[k]; }
      }
      gs_block_tree<SECOND>(a, lgw, g, [&](int pos, int, const GsAcc& r) {
        if (pos != 0) return;
        p.pS[base + c] = r.s;
        if (!SECOND) { p.pN[base + c] = r.n; p.pMn[base + c] = r.mn; p.pMx[base + c] = r.mx; }
      });
    }
    n /= w;
  }
  if (threadIdx.x != 0) return;
  double* o = p.out + ((size_t)g * Q + q) * 5;
  if (!SECOND) { o[0] = p.pN[base]; o[1] = gs_mean(p.pN[base], p.pS[base]); o[3] = p.pMn[base]; o[4] = p.pMx[base]; }
  else o[2] = gs_variance(o[0], p.pS[base]);
}

// ---- time statistics over windows of S8 records (time_stats.cuh; samsim_b200_set_time_stats) --------------------
struct TsParams {
  // snapshot, status and end steps, all in slot order
  const double* snap_sc;   // [SNAPSC_COUNT][ncol_pad]
  const double* snap_arr;  // [SNAPARR_COUNT][LS][ncol_pad]
  const int* in;
  const int64_t* end_of_col;
  const int* map;          // slot_of_col, nullptr = identity
  long long ncol, ncol_pad;
  int LS;
  long long i;             // loop index of the record
  const double* z;
  int nz, nsc, nprof;
  int sc[SAMSIM_SNAPSC_COUNT];     // selected snapshot scalars, ascending
  int prof[SAMSIM_SNAPARR_COUNT];  // selected snapshot arrays, ascending
  double* acc;             // window in progress: [Q][5][ncol_pad] = n, mean, M2, min, max in caller column order
  double* out;             // history slot [Q][5][ncol_pad] when this record closes the window, else nullptr
  bool first;              // the record opens a window: the accumulators are not read
};

// One record of quantity q for caller column c: the Welford update where the column contributes, and on the window's
// closing record the finalised statistics into the history slot instead of the accumulators.
__device__ __forceinline__ void ts_one(const TsParams& p, long long c, int q, bool contributes, double x) {
  const size_t ls = (size_t)p.ncol_pad, base = (size_t)q * SAMSIM_TS_NSTAT * ls + c;
  if (!contributes && !p.first && !p.out) return;  // nothing changes
  TsAcc a = ts_init();
  if (!p.first) a = TsAcc{p.acc[base], p.acc[base + ls], p.acc[base + 2 * ls], p.acc[base + 3 * ls], p.acc[base + 4 * ls]};
  if (contributes) ts_update(a, x);
  if (p.out) {
    double r[SAMSIM_TS_NSTAT];
    ts_finish(a, r);
    for (int s = 0; s < SAMSIM_TS_NSTAT; s++) p.out[base + s * ls] = r[s];
  } else {
    p.acc[base] = a.n; p.acc[base + ls] = a.mean; p.acc[base + 2 * ls] = a.m2; p.acc[base + 3 * ls] = a.mn;
    p.acc[base + 4 * ls] = a.mx;
  }
}

// one thread per caller column: reads its snapshot through slot_of_col (re-binning permutes nothing here)
__global__ void samsim_ts_record_kernel(const TsParams p) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= p.ncol) return;
  const long long s = slot_of(p.map, c);
  const size_t ls = (size_t)p.ncol_pad;
  // failed and finished columns hold stale snapshots
  const bool live = p.in[(size_t)IN_STATUS * ls + s] == 0 && (!p.end_of_col || p.end_of_col[s] >= p.i);
  for (int q = 0; q < p.nsc; q++) ts_one(p, c, q, live, live ? p.snap_sc[(size_t)p.sc[q] * ls + s] : 0.0);
  if (p.nprof == 0) return;
  int reached = 0;  // depths above the column's ice bottom
  if (live) {
    const double* A = p.snap_arr;
    const int LS = p.LS;
    const int na = (int)p.snap_sc[(size_t)SAMSIM_SNAPSC_N_ACTIVE * ls + s];
    auto thick = [&](int k) { return A[((size_t)SAMSIM_SNAPARR_THICK * LS + k) * ls + s]; };
    gs_regrid(thick, na, p.z, p.nz, [&](int j, int k) {
      for (int a = 0; a < p.nprof; a++) ts_one(p, c, p.nsc + a * p.nz + j, true, A[((size_t)p.prof[a] * LS + k) * ls + s]);
      reached = j + 1;
    });
  }
  for (int j = reached; j < p.nz; j++)
    for (int a = 0; a < p.nprof; a++) ts_one(p, c, p.nsc + a * p.nz + j, false, 0.0);
}

// samsim_b200_close_time_window: finalise the window in progress into its history slot, one thread per column
__global__ void samsim_ts_close_kernel(const double* acc, double* out, int Q, long long ncol, long long ncol_pad) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncol) return;
  const size_t ls = (size_t)ncol_pad;
  for (int q = 0; q < Q; q++) {
    const size_t base = (size_t)q * SAMSIM_TS_NSTAT * ls + c;
    const TsAcc a{acc[base], acc[base + ls], acc[base + 2 * ls], acc[base + 3 * ls], acc[base + 4 * ls]};
    double r[SAMSIM_TS_NSTAT];
    ts_finish(a, r);
    for (int s = 0; s < SAMSIM_TS_NSTAT; s++) out[base + s * ls] = r[s];
  }
}

// samsim_b200_get_time_stats: one window's [Q][5][ncol_pad] history -> dst[(cc*Q + q)*5 + s] for columns col0..col0+n-1
__global__ void samsim_ts_get_kernel(const double* win, double* dst, long long ncol_pad, int Q, long long col0, long long n) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * Q * SAMSIM_TS_NSTAT) return;
  const long long cc = t / ((long long)Q * SAMSIM_TS_NSTAT), qs = t % ((long long)Q * SAMSIM_TS_NSTAT);
  dst[t] = win[(size_t)qs * ncol_pad + col0 + cc];
}

__global__ void samsim_count_failed_kernel(const int* in, long long ncol, long long ncol_pad, int* out) {
  const long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (col < ncol && in[(size_t)IN_STATUS * ncol_pad + col] != 0) atomicAdd(out, 1);
}

// ---- KAT kernels -----------------------------------------------------------------------------
static void fill_liquidus(DevCfg& g, int salt_flag) {
  g.salt_flag = salt_flag;
  if (salt_flag == 1) { g.c2 = -18.7; g.c3 = -0.519; g.c4 = -0.00535; g.d2 = -21.4; g.d3x2 = 2.0 * -0.886; g.d4x3 = 3.0 * -0.0170; }  // mo_thermo_functions.f90:321-326 / :393-397
  else { g.c2 = -17.6; g.c3 = -0.389; g.c4 = -0.00362; g.d2 = -17.6; g.d3x2 = 2.0 * -0.389; g.d4x3 = 3.0 * -0.00362; }                // :331-336 / :398-402
}
__global__ void samsim_kat_getT_kernel(int salt_flag, int n, const double* H, const double* S_bu, const double* T_in,
                                       double* T_out, double* phi_out, int* st) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n) return;
  (void)salt_flag;  // the liquidus of salt_flag is in the constant-memory configuration (kat_upload_cfg)
  double T = 0.0, phi = 0.0;
  int status = 0;
  unsigned ev1 = 0;
  getT(H[q], S_bu[q], T_in[q], T, phi, status, ev1);
  // status_out: the STOP code in the low 16 bits; bits 16.. = the EV_GETT_* branch bits (word 1 of the event words)
  T_out[q] = T; phi_out[q] = phi; st[q] = status | (int)(ev1 << 16);
}
__global__ void samsim_kat_scalar_kernel(int fn, int salt_flag, int n, const double* a, const double* b, double* out) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n) return;
  double r;
  switch (fn) {
    case 0: r = S_br_of(a[q]); break;
    case 1: r = S_br_of(a[q], b[q]); break;
    case 2: r = ddT_S_br_of(a[q]); break;
    case 3: r = density_of(a[q], b[q]); break;
    case 4: r = T_freeze_of(a[q], salt_flag); break;
    case 5: r = k_snow_of(a[q], b[q]); break;
    case 6: r = albedo_of(a[q], b[q], 0.1, 0.005, 2); break;
    case 7: r = det_pow(a[q], b[q]); break;
    case 8: r = det_exp(a[q]); break;
    case 9: r = det_sin(a[q]); break;
    default: r = nan("");
  }
  out[q] = r;
}

// FP64 peak: 8 independent fma chains per thread (explicit fma() is not affected by -fmad=false)
__global__ void samsim_fp64_peak_kernel(double* out, int iters, double seed) {
  double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
  const double x = 1.0000001, y = 1e-9;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
      a0 = fma(a0, x, y); a1 = fma(a1, x, y); a2 = fma(a2, x, y); a3 = fma(a3, x, y);
      a4 = fma(a4, x, y); a5 = fma(a5, x, y); a6 = fma(a6, x, y); a7 = fma(a7, x, y);
    }
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CU(call)                                                                             \
  do {                                                                                       \
    cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess) return fail(SAMSIM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

struct samsim_b200_handle_s {
  samsim_config_t cfg;
  DevCfg dcfg;
  int device;
  long long ncol, ncol_pad;
  int LS;
  double* arr = nullptr;
  double* sc = nullptr;
  int* in = nullptr;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_launch = nullptr;  // after the last step kernel: the next owner of the constant-memory configuration waits for it
  bool timed = false;
  // clock
  double time = 0.0;
  long long i = 0;
  int n_time_out = 0, time_counter = 1;
  // forcing
  double* series = nullptr;
  int nsite = 0, nrec = 0;
  int* site_of_col = nullptr;
  double *fscale = nullptr, *foffset = nullptr;
  double* lab = nullptr;
  long long lab_nrec = 0;
  int* set_of_col = nullptr;
  // lab sets: the real length of each set (samsim_b200_set_lab_lengths, else lab_nrec), the set of every column in
  // caller order (empty = all in set 0) and the latest end step of each set's columns (INT64_MIN: the set has none)
  std::vector<int64_t> lab_len, lab_end;
  std::vector<int32_t> set_host;
  // per-column end steps (samsim_b200_set_end_step): device row in slot order (nullptr until the first call) and the
  // host copy in caller order
  int64_t* end_of_col = nullptr;
  std::vector<int64_t> end_host;
  // snapshot
  int snap_mode = SAMSIM_SNAP_NONE;
  double *snap_sc = nullptr, *snap_arr = nullptr;
  // staging
  double* stage = nullptr;
  size_t stage_bytes = 0;
  long long launches = 0;
  int num_sms = 148;
  int n_arr = AR_CORE_COUNT;  // AR_COUNT when tracers are on (cfg.N_bgc > 0)
  // re-binning: slot_of_col[c] = where column c lives, col_of_slot[s] = which column lives in slot s (nullptr = identity)
  int *slot_of_col = nullptr, *col_of_slot = nullptr;
  long long rebin_every = 0, since_rebin = 0, rebins = 0;
  // in-kernel divergence measurement: 4 counters on the device, read back after each step() call into pinned host memory
  unsigned long long* divergence = nullptr;       // device
  unsigned long long* divergence_host = nullptr;  // pinned
  cudaEvent_t ev_div = nullptr;
  bool div_pending = false;
  double rebin_auto_threshold = 0.0;              // 0 = off
  double last_idle_share = 0.0, last_class_split_share = 0.0;
  // group statistics (samsim_b200_set_group_stats): off while gs_ngroup == 0
  int gs_ngroup = 0, gs_Q = 0, gs_nz = 0, gs_nprof = 0, gs_max = 0, gs_held = 0;
  int gs_prof[SAMSIM_SNAPARR_COUNT] = {0};
  uint32_t gs_mask = 0;
  long long gs_npad = 0;
  int gs_nbig = 0;
  int *gs_col = nullptr, *gs_info = nullptr, *gs_big = nullptr;  // gs_big: [3][nbig] group, first tile, log2 size
  double *gs_z = nullptr, *gs_vals = nullptr, *gs_reach = nullptr, *gs_part = nullptr, *gs_hist = nullptr;
  std::vector<double> gs_time;
  std::vector<int64_t> gs_i;
  // time statistics (samsim_b200_set_time_stats): off while ts_Q == 0
  int ts_Q = 0, ts_nsc = 0, ts_nz = 0, ts_nprof = 0, ts_rpw = 0, ts_max = 0, ts_held = 0;
  int ts_cur = 0;  // records in the window in progress
  int ts_sc[SAMSIM_SNAPSC_COUNT] = {0}, ts_prof[SAMSIM_SNAPARR_COUNT] = {0};
  uint32_t ts_mask = 0;  // profile_mask
  double *ts_z = nullptr, *ts_acc = nullptr, *ts_hist = nullptr;
  std::vector<int32_t> ts_nrec;  // [max_windows]
  // [max_windows + 1][2]: time and loop index of the first and last record of each held window, and of the window in
  // progress in row max_windows
  std::vector<double> ts_time;
  std::vector<int64_t> ts_i;
};

// The step kernel reads its configuration from constant memory (samsim_dev_cfg, physics.cuh), one copy per device.
// `g_cfg_owner[device]` is the handle whose DevCfg is there (nullptr: a KAT call overwrote it).  A handle that is not
// the owner waits for the owner's last launch and uploads its own on its stream -- nothing in the common case of one
// handle per device.  One host thread per handle (include/samsim_b200.h); the table itself is guarded by a mutex.
#include <mutex>
static std::mutex g_cfg_mutex;
static samsim_handle_t g_cfg_owner[64] = {nullptr};

static int claim_device_cfg(samsim_handle_t h) {
  std::lock_guard<std::mutex> lock(g_cfg_mutex);
  const int d = h->device & 63;
  if (g_cfg_owner[d] == h) return 0;
  if (g_cfg_owner[d] && g_cfg_owner[d]->ev_launch) CU(cudaStreamWaitEvent(h->stream, g_cfg_owner[d]->ev_launch, 0));
  CU(cudaMemcpyToSymbolAsync(samsim_dev_cfg, &h->dcfg, sizeof(DevCfg), 0, cudaMemcpyHostToDevice, h->stream));
  g_cfg_owner[d] = h;
  return 0;
}
static void release_device_cfg(samsim_handle_t h) {
  std::lock_guard<std::mutex> lock(g_cfg_mutex);
  const int d = h->device & 63;
  if (g_cfg_owner[d] == h) g_cfg_owner[d] = nullptr;
}

static int ensure_stage(samsim_handle_t h, size_t bytes) {
  if (h->stage_bytes >= bytes) return 0;
  if (h->stage) cudaFree(h->stage);
  h->stage = nullptr;
  h->stage_bytes = 0;
  CU(cudaMalloc(&h->stage, bytes));
  h->stage_bytes = bytes;
  return 0;
}

static double host_time_input(int k) { return ((double)(float)k - 1.0) * 3600.0 * 3.0; }

// one per-column row <-> host vector; straight copies while the columns are in their original order
template <typename T>
static int vec_set(samsim_handle_t h, T* row, const T* host, int32_t col0, int32_t n) {
  if (n == 0) return 0;
  if (!h->slot_of_col) {
    CU(cudaMemcpyAsync(row + col0, host, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, h->stream));
  } else {
    int rc;
    if ((rc = ensure_stage(h, (size_t)n * sizeof(T)))) return rc;
    CU(cudaMemcpyAsync(h->stage, host, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    samsim_vec_set_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(row, (const T*)h->stage, col0, n, h->slot_of_col);
    CU(cudaGetLastError());
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}
template <typename T>
static int vec_get(samsim_handle_t h, const T* row, T* host, int32_t col0, int32_t n) {
  if (n == 0) return 0;
  if (!h->slot_of_col) {
    CU(cudaMemcpyAsync(host, row + col0, (size_t)n * sizeof(T), cudaMemcpyDeviceToHost, h->stream));
  } else {
    int rc;
    if ((rc = ensure_stage(h, (size_t)n * sizeof(T)))) return rc;
    samsim_vec_get_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(row, (T*)h->stage, col0, n, h->slot_of_col);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(host, h->stage, (size_t)n * sizeof(T), cudaMemcpyDeviceToHost, h->stream));
  }
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

// rows[r][s] <- rows[r][order[s]] for nrows rows of ncol_pad elements (tmp holds nrows*ncol_pad elements)
template <typename T>
static int permute_rows(samsim_handle_t h, T* rows, int nrows, const int* order, void* tmp) {
  if (!rows || nrows <= 0) return 0;
  const long long total = (long long)nrows * h->ncol_pad;
  samsim_permute_rows_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(rows, (T*)tmp, h->ncol, h->ncol_pad, nrows, order);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(rows, tmp, (size_t)total * sizeof(T), cudaMemcpyDeviceToDevice, h->stream));
  return 0;
}
static size_t permute_tmp_bytes(samsim_handle_t h) {
  int rows = h->LS;
  if (rows < SC_COUNT) rows = SC_COUNT;
  if (rows < SAMSIM_SNAPSC_COUNT) rows = SAMSIM_SNAPSC_COUNT;
  return (size_t)rows * h->ncol_pad * sizeof(double);
}
// per-column forcing vectors arrive in column order; bring them into slot order when the handle is re-binned
template <typename T>
static int to_slot_order(samsim_handle_t h, T* rows, int nrows) {
  if (!h->col_of_slot || !rows) return 0;
  void* tmp = nullptr;
  CU(cudaMalloc(&tmp, permute_tmp_bytes(h)));
  int rc = permute_rows<T>(h, rows, nrows, h->col_of_slot, tmp);
  cudaStreamSynchronize(h->stream);
  cudaFree(tmp);
  return rc;
}

static void gs_free(samsim_handle_t h) {
  cudaFree(h->gs_col); cudaFree(h->gs_info); cudaFree(h->gs_big); cudaFree(h->gs_z); cudaFree(h->gs_vals);
  cudaFree(h->gs_reach); cudaFree(h->gs_part); cudaFree(h->gs_hist);
  h->gs_col = h->gs_info = h->gs_big = nullptr;
  h->gs_z = h->gs_vals = h->gs_reach = h->gs_part = h->gs_hist = nullptr;
  h->gs_ngroup = h->gs_Q = h->gs_nz = h->gs_nprof = h->gs_max = h->gs_held = h->gs_nbig = 0;
  h->gs_mask = 0;
  h->gs_npad = 0;
  h->gs_time.clear();
  h->gs_i.clear();
}

// Queue the statistics of the record just written by the last step kernel (loop index h->i, model time `time`) into
// history slot gs_held.  Five kernels on the handle's stream, no host synchronisation.
static int gs_record(samsim_handle_t h, double time) {
  GsParams p;
  memset(&p, 0, sizeof p);
  p.snap_sc = h->snap_sc; p.snap_arr = h->snap_arr; p.in = h->in; p.end_of_col = h->end_of_col; p.map = h->slot_of_col;
  p.ncol_pad = h->ncol_pad; p.LS = h->LS; p.i = h->i;
  p.col = h->gs_col; p.info = h->gs_info; p.npad = h->gs_npad;
  p.z = h->gs_z; p.nz = h->gs_nz; p.nprof = h->gs_nprof; p.Q = h->gs_Q;
  for (int a = 0; a < h->gs_nprof; a++) p.prof[a] = h->gs_prof[a];
  p.vals = h->gs_vals; p.reach = h->gs_reach;
  const size_t npart = (size_t)h->gs_Q * (h->gs_npad / SAMSIM_GS_TILE);
  p.pS = h->gs_part; p.pN = p.pS + npart; p.pMn = p.pN + npart; p.pMx = p.pMn + npart;
  p.big_group = h->gs_big;
  p.out = h->gs_hist + (size_t)h->gs_held * h->gs_ngroup * h->gs_Q * 5;
  const unsigned ntile = (unsigned)(h->gs_npad / SAMSIM_GS_TILE);
  samsim_gs_gather_kernel<<<(unsigned)((h->gs_npad + 255) / 256), 256, 0, h->stream>>>(p);
  const dim3 big((unsigned)h->gs_nbig, (unsigned)h->gs_Q);
  samsim_gs_tile_kernel<false><<<ntile, SAMSIM_GS_TILE, 0, h->stream>>>(p);
  if (h->gs_nbig) samsim_gs_final_kernel<false><<<big, SAMSIM_GS_TILE, 0, h->stream>>>(p, h->gs_big + h->gs_nbig, h->gs_big + 2 * h->gs_nbig);
  samsim_gs_tile_kernel<true><<<ntile, SAMSIM_GS_TILE, 0, h->stream>>>(p);
  if (h->gs_nbig) samsim_gs_final_kernel<true><<<big, SAMSIM_GS_TILE, 0, h->stream>>>(p, h->gs_big + h->gs_nbig, h->gs_big + 2 * h->gs_nbig);
  CU(cudaGetLastError());
  h->gs_time[(size_t)h->gs_held] = time;
  h->gs_i[(size_t)h->gs_held] = h->i;
  h->gs_held++;
  return 0;
}

// records that `nsteps` steps from the current clock write (output steps: i == 1 and every i_time_out+1 steps)
static int64_t records_in(samsim_handle_t h, int64_t nsteps) {
  return ts_records_in(h->i, h->n_time_out, h->cfg.i_time_out, nsteps);
}

static void ts_free(samsim_handle_t h) {
  cudaFree(h->ts_z); cudaFree(h->ts_acc); cudaFree(h->ts_hist);
  h->ts_z = h->ts_acc = h->ts_hist = nullptr;
  h->ts_Q = h->ts_nsc = h->ts_nz = h->ts_nprof = h->ts_rpw = h->ts_max = h->ts_held = h->ts_cur = 0;
  h->ts_mask = 0;
  h->ts_nrec.clear();
  h->ts_time.clear();
  h->ts_i.clear();
}

// the window in progress becomes history slot ts_held (its statistics were written there by the kernels)
static void ts_window_done(samsim_handle_t h) {
  const size_t w = (size_t)h->ts_held, cur = (size_t)h->ts_max;
  h->ts_nrec[w] = h->ts_cur;
  for (int k = 0; k < 2; k++) {
    h->ts_time[2 * w + k] = h->ts_time[2 * cur + k];
    h->ts_i[2 * w + k] = h->ts_i[2 * cur + k];
  }
  h->ts_held++;
  h->ts_cur = 0;
}

// Queue the record just written by the last step kernel (loop index h->i, model time `time`) into the window in
// progress; on its closing record the same kernel writes history slot ts_held.  No host synchronisation.
static int ts_record(samsim_handle_t h, double time) {
  TsParams p;
  memset(&p, 0, sizeof p);
  p.snap_sc = h->snap_sc; p.snap_arr = h->snap_arr; p.in = h->in; p.end_of_col = h->end_of_col; p.map = h->slot_of_col;
  p.ncol = h->ncol; p.ncol_pad = h->ncol_pad; p.LS = h->LS; p.i = h->i;
  p.z = h->ts_z; p.nz = h->ts_nz; p.nsc = h->ts_nsc; p.nprof = h->ts_nprof;
  for (int q = 0; q < h->ts_nsc; q++) p.sc[q] = h->ts_sc[q];
  for (int a = 0; a < h->ts_nprof; a++) p.prof[a] = h->ts_prof[a];
  p.acc = h->ts_acc;
  p.first = (h->ts_cur == 0);
  const bool closes = h->ts_rpw > 0 && h->ts_cur + 1 == h->ts_rpw;
  p.out = closes ? h->ts_hist + (size_t)h->ts_held * h->ts_Q * SAMSIM_TS_NSTAT * h->ncol_pad : nullptr;
  samsim_ts_record_kernel<<<(unsigned)((h->ncol + 255) / 256), 256, 0, h->stream>>>(p);
  CU(cudaGetLastError());
  const size_t cur = (size_t)h->ts_max;
  if (p.first) { h->ts_time[2 * cur] = time; h->ts_i[2 * cur] = h->i; }
  h->ts_time[2 * cur + 1] = time;
  h->ts_i[2 * cur + 1] = h->i;
  h->ts_cur++;
  if (closes) ts_window_done(h);
  return 0;
}

extern "C" {

const char* samsim_b200_last_error(void) { return g_err.c_str(); }
const char* samsim_b200_version(void) { return "samsim_b200 0.1 (sm_100a, fp64, fmad=false)"; }

int samsim_b200_create(const samsim_config_t* cfg, int32_t ncol, int32_t device, samsim_handle_t* out) {
  if (!cfg || !out || ncol < 1) return fail(SAMSIM_ERR_ARG, "create: bad argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
    return fail(SAMSIM_ERR_NO_DEVICE, "no CUDA device: samsim_b200 has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(SAMSIM_ERR_ARG, "create: bad device index");
  if (cfg->Nlayer < 3 || cfg->Nlayer != cfg->N_top + cfg->N_middle + cfg->N_bottom || cfg->N_top < 3)
    return fail(SAMSIM_ERR_CONFIG, "Nlayer must equal N_top+N_middle+N_bottom with N_top >= 3 (mo_init.f90:2014-2017)");
  if (!(cfg->salt_flag == 1 || cfg->salt_flag == 2)) return fail(SAMSIM_ERR_CONFIG, "salt_flag must be 1 or 2");
  if (cfg->N_bgc < 0 || cfg->N_bgc > 2) return fail(SAMSIM_ERR_CONFIG, "N_bgc must be 0 (bgc_flag 1), 1 or 2");
  if (!(cfg->dt > 0.0) || !(cfg->thick_0 > 0.0)) return fail(SAMSIM_ERR_CONFIG, "dt and thick_0 must be positive");
  CU(cudaSetDevice(device));
  samsim_handle_t h = new samsim_b200_handle_s();
  {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) h->num_sms = sms;
  }
  h->cfg = *cfg;
  h->device = device;
  h->ncol = ncol;
  h->ncol_pad = ((long long)ncol + SAMSIM_BLOCK - 1) / SAMSIM_BLOCK * SAMSIM_BLOCK;
  h->LS = cfg->Nlayer + 2;
  h->n_arr = (cfg->N_bgc > 0) ? AR_COUNT : AR_CORE_COUNT;
  // (32-bit index arithmetic is confined to one tile: (Nlayer+2)*n_arr*32 elements; no limit on the column count
  // other than memory)
  if ((unsigned long long)h->n_arr * h->LS * SAMSIM_TILE >= (1ull << 31)) {
    delete h;
    return fail(SAMSIM_ERR_ARG, "create: Nlayer too large for the 32-bit in-tile index");
  }
  DevCfg& d = h->dcfg;
  memset(&d, 0, sizeof d);
  d.testcase = cfg->testcase; d.Nlayer = cfg->Nlayer; d.N_top = cfg->N_top; d.N_middle = cfg->N_middle; d.N_bottom = cfg->N_bottom;
  d.atmoflux_flag = cfg->atmoflux_flag; d.grav_flag = cfg->grav_flag; d.prescribe_flag = cfg->prescribe_flag;
  d.grav_heat_flag = cfg->grav_heat_flag; d.flush_heat_flag = cfg->flush_heat_flag; d.turb_flag = cfg->turb_flag;
  d.salt_flag = cfg->salt_flag; d.boundflux_flag = cfg->boundflux_flag; d.flush_flag = cfg->flush_flag;
  d.flood_flag = cfg->flood_flag; d.bottom_flag = cfg->bottom_flag; d.precip_flag = cfg->precip_flag;
  d.harmonic_flag = cfg->harmonic_flag; d.tank_flag = cfg->tank_flag; d.albedo_flag = cfg->albedo_flag;
  d.lab_snow_flag = cfg->lab_snow_flag; d.freeboard_snow_flag = cfg->freeboard_snow_flag;
  d.snow_flush_flag = cfg->snow_flush_flag; d.snow_precip_flag = cfg->snow_precip_flag;
  d.i_time_out = cfg->i_time_out;
  d.n_bgc = cfg->N_bgc;
  d.dt = cfg->dt; d.thick_0 = cfg->thick_0; d.thick_min = cfg->thick_min; d.time_out = cfg->time_out;
  d.alpha_flux_instable = cfg->alpha_flux_instable; d.alpha_flux_stable = cfg->alpha_flux_stable; d.m_total = cfg->m_total;
  d.max_flux_plate = cfg->max_flux_plate; d.k_snow_flush = cfg->k_snow_flush; d.k_styropor = cfg->k_styropor;
  fill_liquidus(d, cfg->salt_flag);
  // prefetch distance: 2 layers (large batches: 70.8 M column-steps/s against 69.5 at 4 and 64.7 at 12 in round 1; small
  // batches are bound by the dependent FP64 chains of their few warps, not by load latency: 2 / 6 / 12 / 24 layers all
  // give 31.2 M column-steps/s on 10,000 testcase-1 columns, profiles/README.md)
  d.pf = 2;
  const size_t narr = (size_t)h->n_arr * h->LS * h->ncol_pad;
  cudaError_t e;
  if ((e = cudaMalloc(&h->arr, narr * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->sc, (size_t)SC_COUNT * h->ncol_pad * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->in, (size_t)IN_COUNT * h->ncol_pad * sizeof(int))) != cudaSuccess) {
    samsim_b200_destroy(h);
    return fail(SAMSIM_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  }
  cudaMemset(h->arr, 0, narr * sizeof(double));
  cudaMemset(h->sc, 0, (size_t)SC_COUNT * h->ncol_pad * sizeof(double));
  cudaMemset(h->in, 0, (size_t)IN_COUNT * h->ncol_pad * sizeof(int));
  cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  cudaEventCreate(&h->ev0);
  cudaEventCreate(&h->ev1);
  cudaEventCreateWithFlags(&h->ev_launch, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->ev_div, cudaEventDisableTiming);
  if (cudaMalloc(&h->divergence, 4 * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMallocHost(&h->divergence_host, 4 * sizeof(unsigned long long)) != cudaSuccess) {
    samsim_b200_destroy(h);
    return fail(SAMSIM_ERR_CUDA, "cudaMalloc: divergence counters");
  }
  memset(h->divergence_host, 0, 4 * sizeof(unsigned long long));
  *out = h;
  return SAMSIM_OK;
}

void samsim_b200_destroy(samsim_handle_t h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  release_device_cfg(h);
  if (h->ev_launch) cudaEventDestroy(h->ev_launch);
  if (h->ev_div) cudaEventDestroy(h->ev_div);
  cudaFree(h->divergence);
  if (h->divergence_host) cudaFreeHost(h->divergence_host);
  cudaFree(h->arr); cudaFree(h->sc); cudaFree(h->in); cudaFree(h->series); cudaFree(h->site_of_col);
  cudaFree(h->fscale); cudaFree(h->foffset); cudaFree(h->lab); cudaFree(h->set_of_col); cudaFree(h->snap_sc);
  cudaFree(h->snap_arr); cudaFree(h->stage); cudaFree(h->slot_of_col); cudaFree(h->col_of_slot); cudaFree(h->end_of_col);
  gs_free(h);
  ts_free(h);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

// public array id -> slot in the device buffer (the tracer arrays sit behind the scratch arrays)
static inline int arr_slot(int32_t id) { return (id < AR_STATE_COUNT) ? id : AR_BGC1 + (id - AR_STATE_COUNT); }

int32_t samsim_b200_array_extent(samsim_handle_t h, int32_t id) {
  if (!h || id < 0 || id >= SAMSIM_ARR_COUNT) return -1;
  if (id >= SAMSIM_ARR_BGC_ABS1) return (id - SAMSIM_ARR_BGC_ABS1 < h->cfg.N_bgc) ? h->cfg.Nlayer : -1;
  if (id == SAMSIM_ARR_RAY) return h->cfg.Nlayer - 1;
  if (id == SAMSIM_ARR_FL_Q) return h->cfg.Nlayer + 1;
  return h->cfg.Nlayer;
}

static int check_cols(samsim_handle_t h, int32_t col0, int32_t n) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (col0 < 0 || n < 0 || (long long)col0 + n > h->ncol) return fail(SAMSIM_ERR_ARG, "column range out of bounds");
  return 0;
}

int samsim_b200_set_array(samsim_handle_t h, int32_t id, const double* host, int32_t col0, int32_t n) {
  int rc = check_cols(h, col0, n);
  if (rc) return rc;
  const int ext = samsim_b200_array_extent(h, id);
  if (ext < 0 || !host) return fail(SAMSIM_ERR_ARG, "set_array: bad id or null pointer");
  if (n == 0) return 0;
  CU(cudaSetDevice(h->device));
  const size_t bytes = (size_t)n * ext * sizeof(double);
  if ((rc = ensure_stage(h, bytes))) return rc;
  CU(cudaMemcpyAsync(h->stage, host, bytes, cudaMemcpyHostToDevice, h->stream));
  const long long total = (long long)n * ext;
  samsim_scatter_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(h->arr, h->stage, h->LS, h->n_arr, arr_slot(id), ext, col0, n, h->slot_of_col);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int samsim_b200_get_array(samsim_handle_t h, int32_t id, double* host, int32_t col0, int32_t n) {
  int rc = check_cols(h, col0, n);
  if (rc) return rc;
  const int ext = samsim_b200_array_extent(h, id);
  if (ext < 0 || !host) return fail(SAMSIM_ERR_ARG, "get_array: bad id or null pointer");
  if (n == 0) return 0;
  CU(cudaSetDevice(h->device));
  const size_t bytes = (size_t)n * ext * sizeof(double);
  if ((rc = ensure_stage(h, bytes))) return rc;
  const long long total = (long long)n * ext;
  samsim_state_gather_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(h->arr, h->stage, h->LS, h->n_arr, arr_slot(id), ext, col0, n, h->slot_of_col);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(host, h->stage, bytes, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int samsim_b200_set_scalar(samsim_handle_t h, int32_t id, const double* host, int32_t col0, int32_t n) {
  int rc = check_cols(h, col0, n);
  if (rc) return rc;
  if (id < 0 || id >= SAMSIM_SC_COUNT || !host) return fail(SAMSIM_ERR_ARG, "set_scalar: bad id or null pointer");
  CU(cudaSetDevice(h->device));
  return vec_set<double>(h, h->sc + (size_t)id * h->ncol_pad, host, col0, n);
}
int samsim_b200_get_scalar(samsim_handle_t h, int32_t id, double* host, int32_t col0, int32_t n) {
  int rc = check_cols(h, col0, n);
  if (rc) return rc;
  if (id < 0 || id >= SAMSIM_SC_COUNT || !host) return fail(SAMSIM_ERR_ARG, "get_scalar: bad id or null pointer");
  CU(cudaSetDevice(h->device));
  return vec_get<double>(h, h->sc + (size_t)id * h->ncol_pad, host, col0, n);
}
int samsim_b200_set_int(samsim_handle_t h, int32_t id, const int32_t* host, int32_t col0, int32_t n) {
  int rc = check_cols(h, col0, n);
  if (rc) return rc;
  if (id < 0 || id >= SAMSIM_INT_COUNT || !host) return fail(SAMSIM_ERR_ARG, "set_int: bad id or null pointer");
  CU(cudaSetDevice(h->device));
  return vec_set<int>(h, h->in + (size_t)id * h->ncol_pad, host, col0, n);
}
int samsim_b200_get_int(samsim_handle_t h, int32_t id, int32_t* host, int32_t col0, int32_t n) {
  int rc = check_cols(h, col0, n);
  if (rc) return rc;
  if (id < 0 || id >= SAMSIM_INT_COUNT || !host) return fail(SAMSIM_ERR_ARG, "get_int: bad id or null pointer");
  CU(cudaSetDevice(h->device));
  return vec_get<int>(h, h->in + (size_t)id * h->ncol_pad, host, col0, n);
}

int samsim_b200_broadcast_column(samsim_handle_t h, int32_t src, int32_t col0, int32_t n) {
  int rc = check_cols(h, col0, n);
  if (rc) return rc;
  if (src < 0 || src >= h->ncol) return fail(SAMSIM_ERR_ARG, "broadcast: bad source column");
  if (n == 0) return 0;
  CU(cudaSetDevice(h->device));
  samsim_broadcast_kernel<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>(h->arr, h->sc, h->in, h->ncol_pad, h->LS, src, col0, n, h->slot_of_col, h->n_arr);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int samsim_b200_set_clock(samsim_handle_t h, double time, int64_t i, int32_t n_time_out, int32_t time_counter) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (time_counter < 1) return fail(SAMSIM_ERR_ARG, "time_counter is 1-based");
  if (i < 0 || n_time_out < 0 || n_time_out > h->cfg.i_time_out)
    return fail(SAMSIM_ERR_ARG, "set_clock: need i >= 0 and 0 <= n_time_out <= i_time_out (mo_grotz.f90:340: a record is written when n_time_out == i_time_out)");
  h->time = time; h->i = i; h->n_time_out = n_time_out; h->time_counter = time_counter;
  return 0;
}
int samsim_b200_get_clock(samsim_handle_t h, double* time, int64_t* i, int32_t* n_time_out, int32_t* time_counter) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (time) *time = h->time;
  if (i) *i = h->i;
  if (n_time_out) *n_time_out = h->n_time_out;
  if (time_counter) *time_counter = h->time_counter;
  return 0;
}

static void drop_forcing(samsim_handle_t h) {
  cudaFree(h->series); cudaFree(h->site_of_col); cudaFree(h->fscale); cudaFree(h->foffset);
  h->series = nullptr; h->site_of_col = nullptr; h->fscale = nullptr; h->foffset = nullptr;
  h->nsite = h->nrec = 0;
}

static int upload_forcing(samsim_handle_t h, int32_t nsite, int32_t nrec, const double* series, const int32_t* site_of_col,
                          const double* scale, const double* offset) {
  const size_t nb = (size_t)nsite * 4 * (size_t)nrec * sizeof(double);
  CU(cudaMalloc(&h->series, nb));
  CU(cudaMemcpy(h->series, series, nb, cudaMemcpyHostToDevice));
  h->nsite = nsite; h->nrec = nrec;
  if (site_of_col) {
    CU(cudaMalloc(&h->site_of_col, (size_t)h->ncol_pad * sizeof(int)));
    CU(cudaMemset(h->site_of_col, 0, (size_t)h->ncol_pad * sizeof(int)));
    CU(cudaMemcpy(h->site_of_col, site_of_col, (size_t)h->ncol * sizeof(int), cudaMemcpyHostToDevice));
    int rc = to_slot_order<int>(h, h->site_of_col, 1);
    if (rc) return rc;
  }
  for (int w = 0; w < 2; w++) {
    const double* src = w ? offset : scale;
    if (!src) continue;
    double** dst = w ? &h->foffset : &h->fscale;
    CU(cudaMalloc(dst, (size_t)4 * h->ncol_pad * sizeof(double)));
    CU(cudaMemset(*dst, 0, (size_t)4 * h->ncol_pad * sizeof(double)));
    CU(cudaMemcpy2D(*dst, (size_t)h->ncol_pad * sizeof(double), src, (size_t)h->ncol * sizeof(double), (size_t)h->ncol * sizeof(double), 4, cudaMemcpyHostToDevice));
    int rc = to_slot_order<double>(h, *dst, 4);
    if (rc) return rc;
  }
  return 0;
}

int samsim_b200_set_forcing(samsim_handle_t h, int32_t nsite, int32_t nrec, const double* series, const int32_t* site_of_col,
                            const double* scale, const double* offset) {
  if (!h || !series || nsite < 1 || nrec < 2) return fail(SAMSIM_ERR_ARG, "set_forcing: bad argument");
  if (site_of_col)  // validate everything before the tables of the previous call are replaced
    for (long long c = 0; c < h->ncol; c++)
      if (site_of_col[c] < 0 || site_of_col[c] >= nsite) return fail(SAMSIM_ERR_ARG, "set_forcing: site index out of range");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));  // a launch in flight may still read the old tables
  drop_forcing(h);
  const int rc = upload_forcing(h, nsite, nrec, series, site_of_col, scale, offset);
  if (rc) {  // e.g. a table larger than the free device memory: the handle is left without forcing
    drop_forcing(h);
    cudaGetLastError();  // an allocation failure is not sticky; keep it from surfacing at the next launch check
  }
  return rc;
}

int samsim_b200_update_forcing(samsim_handle_t h, const double* series) {
  if (!h || !series) return fail(SAMSIM_ERR_ARG, "update_forcing: bad argument");
  if (!h->series) return fail(SAMSIM_ERR_STATE, "update_forcing: call samsim_b200_set_forcing first");
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpyAsync(h->series, series, (size_t)h->nsite * 4 * h->nrec * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  return 0;
}

int samsim_b200_update_forcing_records(samsim_handle_t h, int32_t rec0, int32_t n, const double* series) {
  if (!h || !series) return fail(SAMSIM_ERR_ARG, "update_forcing_records: bad argument");
  if (!h->series) return fail(SAMSIM_ERR_STATE, "update_forcing_records: call samsim_b200_set_forcing first");
  if (n < 1 || rec0 < 1 || (int64_t)rec0 + n - 1 > h->nrec)
    return fail(SAMSIM_ERR_ARG, "update_forcing_records: records rec0 .. rec0+n-1 must lie in 1..nrec");
  CU(cudaSetDevice(h->device));
  // one row of n records per (site, kind): source rows are n apart, table rows nrec apart
  CU(cudaMemcpy2DAsync(h->series + (rec0 - 1), (size_t)h->nrec * sizeof(double), series, (size_t)n * sizeof(double),
                       (size_t)n * sizeof(double), (size_t)h->nsite * 4, cudaMemcpyHostToDevice, h->stream));
  return 0;
}

// latest end step of the columns of each lab set: only the sets of running columns bound a launch (samsim_b200_step)
static void update_lab_end(samsim_handle_t h) {
  h->lab_end.assign(h->lab_len.size(), INT64_MIN);
  if (h->lab_end.empty()) return;
  for (long long c = 0; c < h->ncol; c++) {
    int64_t& e = h->lab_end[h->set_host.empty() ? 0 : h->set_host[c]];
    e = std::max(e, h->end_host.empty() ? INT64_MAX : h->end_host[c]);
  }
}

int samsim_b200_set_lab_forcing(samsim_handle_t h, int32_t nset, int64_t nrec, const double* series, const int32_t* set_of_col) {
  if (!h || !series || nset < 1 || nrec < 1) return fail(SAMSIM_ERR_ARG, "set_lab_forcing: bad argument");
  if (set_of_col)
    for (long long c = 0; c < h->ncol; c++)
      if (set_of_col[c] < 0 || set_of_col[c] >= nset) return fail(SAMSIM_ERR_ARG, "set_lab_forcing: set index out of range");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  cudaFree(h->lab); cudaFree(h->set_of_col);
  h->lab = nullptr; h->set_of_col = nullptr;
  const size_t nb = (size_t)nset * 4 * nrec * sizeof(double);
  CU(cudaMalloc(&h->lab, nb));
  CU(cudaMemcpy(h->lab, series, nb, cudaMemcpyHostToDevice));
  if (h->cfg.snow_precip_flag == 0) {  // mo_grotz.f90:147-149
    for (int s = 0; s < nset; s++) CU(cudaMemset(h->lab + ((size_t)s * 4 + 1) * nrec, 0, (size_t)nrec * sizeof(double)));
  }
  h->lab_nrec = nrec;
  h->lab_len.assign((size_t)nset, nrec);
  if (set_of_col) h->set_host.assign(set_of_col, set_of_col + h->ncol);
  else h->set_host.clear();
  update_lab_end(h);
  if (set_of_col) {
    CU(cudaMalloc(&h->set_of_col, (size_t)h->ncol_pad * sizeof(int)));
    CU(cudaMemset(h->set_of_col, 0, (size_t)h->ncol_pad * sizeof(int)));
    CU(cudaMemcpy(h->set_of_col, set_of_col, (size_t)h->ncol * sizeof(int), cudaMemcpyHostToDevice));
    int rc = to_slot_order<int>(h, h->set_of_col, 1);
    if (rc) return rc;
  }
  return 0;
}

int samsim_b200_set_lab_lengths(samsim_handle_t h, int32_t nset, const int64_t* nrec_of_set) {
  if (!h || !nrec_of_set) return fail(SAMSIM_ERR_ARG, "set_lab_lengths: bad argument");
  if (!h->lab) return fail(SAMSIM_ERR_STATE, "set_lab_lengths: call samsim_b200_set_lab_forcing first");
  if (nset != (int32_t)h->lab_len.size()) return fail(SAMSIM_ERR_ARG, "set_lab_lengths: nset differs from the last samsim_b200_set_lab_forcing");
  for (int32_t s = 0; s < nset; s++)
    if (nrec_of_set[s] < 1 || nrec_of_set[s] > h->lab_nrec) return fail(SAMSIM_ERR_ARG, "set_lab_lengths: every length must be in 1..nrec");
  h->lab_len.assign(nrec_of_set, nrec_of_set + nset);
  return 0;
}

int samsim_b200_set_end_step(samsim_handle_t h, const int64_t* end_i, int32_t col0, int32_t n) {
  int rc = check_cols(h, col0, n);
  if (rc) return rc;
  if (n > 0 && !end_i) return fail(SAMSIM_ERR_ARG, "set_end_step: null pointer");
  for (int32_t q = 0; q < n; q++)
    if (end_i[q] < 0) return fail(SAMSIM_ERR_ARG, "set_end_step: end steps must be >= 0 (INT64_MAX = no end)");
  if (n == 0) return 0;
  CU(cudaSetDevice(h->device));
  if (!h->end_of_col) {  // every column starts without an end, whatever the slot order
    const std::vector<int64_t> none((size_t)h->ncol_pad, INT64_MAX);
    CU(cudaMalloc(&h->end_of_col, none.size() * sizeof(int64_t)));
    CU(cudaMemcpyAsync(h->end_of_col, none.data(), none.size() * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    h->end_host.assign((size_t)h->ncol, INT64_MAX);
  }
  if ((rc = vec_set<int64_t>(h, h->end_of_col, end_i, col0, n))) return rc;
  std::copy(end_i, end_i + n, h->end_host.begin() + col0);
  update_lab_end(h);
  return 0;
}

// advance the host copy of the clock by one step exactly like the device does
// (true: the step wrote an output record)
static inline bool clock_tick(samsim_handle_t h) {
  h->i += 1;
  const bool out = (h->n_time_out == h->cfg.i_time_out || h->i == 1);
  if (h->cfg.atmoflux_flag == 2 && h->time > host_time_input(h->time_counter)) h->time_counter += 1;
  h->n_time_out = out ? 0 : h->n_time_out + 1;
  h->time = h->time + h->cfg.dt;
  return out;
}

// Divergence of the last launch (measured in the kernel with warp reductions / ballots): fold the counters into the
// handle and, when automatic re-binning is on and idle lane-layers exceed the threshold, re-bin the columns.
static int collect_divergence(samsim_handle_t h, bool may_rebin) {
  if (!h->div_pending) return 0;
  CU(cudaEventSynchronize(h->ev_div));
  h->div_pending = false;
  const unsigned long long* d = h->divergence_host;
  h->last_idle_share = d[1] ? (double)d[0] / (double)d[1] : 0.0;
  h->last_class_split_share = d[3] ? (double)d[2] / (double)d[3] : 0.0;
  if (may_rebin && h->rebin_auto_threshold > 0.0 &&
      (h->last_idle_share > h->rebin_auto_threshold || h->last_class_split_share > 4.0 * h->rebin_auto_threshold))
    return samsim_b200_rebin(h, nullptr);
  return 0;
}

int samsim_b200_set_rebin_auto(samsim_handle_t h, double idle_share_threshold) {
  if (!h || !(idle_share_threshold >= 0.0) || idle_share_threshold >= 1.0) return fail(SAMSIM_ERR_ARG, "set_rebin_auto: threshold in [0, 1)");
  h->rebin_auto_threshold = idle_share_threshold;
  return 0;
}

int samsim_b200_get_divergence(samsim_handle_t h, double* idle_lane_layer_share, double* snow_class_split_warp_share, int64_t* rebins) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  int rc = collect_divergence(h, /*may_rebin=*/false);
  if (rc) return rc;
  if (idle_lane_layer_share) *idle_lane_layer_share = h->last_idle_share;
  if (snow_class_split_warp_share) *snow_class_split_warp_share = h->last_class_split_share;
  if (rebins) *rebins = h->rebins;
  return 0;
}

int64_t samsim_b200_steps_to_next_output(samsim_handle_t h) {
  if (!h) return -1;
  if (h->i == 0) return 1;
  return (int64_t)(h->cfg.i_time_out - h->n_time_out) + 1;
}

int samsim_b200_step(samsim_handle_t h, int64_t nsteps) {
  if (!h || nsteps < 0) return fail(SAMSIM_ERR_ARG, "step: bad argument");
  if (nsteps == 0) return 0;
  const bool need_forcing = (h->cfg.atmoflux_flag == 2);
  const bool tc8 = (h->cfg.testcase == 8);  // T_top = Tinput(FLOOR(1 + time/60)) while time < 475200 s (mo_grotz.f90:539-544)
  const bool need_lab = tc8 || h->cfg.testcase == 111 || (h->cfg.testcase >= 101 && h->cfg.testcase <= 105) ||
                        (h->cfg.boundflux_flag == 3 && h->cfg.lab_snow_flag == 1);  // 111: T_top = Ttop_input(FLOOR(1 + time/dt))
  if (need_forcing && !h->series) return fail(SAMSIM_ERR_STATE, "step: atmoflux_flag 2 needs samsim_b200_set_forcing first");
  if (need_lab && !h->lab) return fail(SAMSIM_ERR_STATE, "step: lab testcases need samsim_b200_set_lab_forcing first");
  if (h->gs_ngroup > 0 && (int64_t)h->gs_held + records_in(h, nsteps) > h->gs_max)
    return fail(SAMSIM_ERR_STATE, "step: the call writes more output records than the group statistics history can hold "
                                  "(samsim_b200_get_group_stats / _clear_group_stats, or a larger max_records)");
  if (h->ts_Q > 0 && ts_windows_completed(h->ts_rpw, h->ts_cur, records_in(h, nsteps)) > (int64_t)h->ts_max - h->ts_held)
    return fail(SAMSIM_ERR_STATE, "step: the call completes more windows than the time statistics history can hold "
                                  "(samsim_b200_get_time_stats / _clear_time_stats, or a larger max_windows)");
  CU(cudaSetDevice(h->device));
  {
    int rc = collect_divergence(h, /*may_rebin=*/true);  // the previous call's measurement decides about re-binning now
    if (rc) return rc;
  }
  CU(cudaMemsetAsync(h->divergence, 0, 4 * sizeof(unsigned long long), h->stream));
  CU(cudaEventRecord(h->ev0, h->stream));
  int64_t left = nsteps;
  while (left > 0) {
    // how many steps fit the staged forcing window?
    KParams p;
    memset(&p, 0, sizeof p);
    p.arr = h->arr; p.n_arr = h->n_arr; p.sc = h->sc; p.in = h->in;
    p.ncol = h->ncol; p.ncol_pad = h->ncol_pad; p.LS = h->LS;
    p.time = h->time; p.i = h->i; p.n_time_out = h->n_time_out; p.time_counter = h->time_counter;
    int64_t chunk = left;
    if (chunk > 1000000) chunk = 1000000;
    if (h->rebin_every > 0 && chunk > h->rebin_every - h->since_rebin) chunk = h->rebin_every - h->since_rebin;
    // group and time statistics read the snapshot, status and end steps of each record: no launch runs past an
    // output step
    if ((h->gs_ngroup > 0 || h->ts_Q > 0) && chunk > samsim_b200_steps_to_next_output(h))
      chunk = samsim_b200_steps_to_next_output(h);
    if (need_forcing) {
      // simulate the clock to find the records the launch touches
      const int tc0 = h->time_counter;
      double t = h->time;
      int tc = tc0;
      int64_t s = 0;
      const int first = (tc0 > 1) ? tc0 - 1 : 1;
      for (; s < chunk; s++) {
        int tcn = tc;
        if (t > host_time_input(tcn)) tcn++;
        if (tcn - first + 1 > SAMSIM_MAXWIN) break;
        if (tcn > h->nrec) {
          if (s == 0) return fail(SAMSIM_ERR_STATE, "step: forcing series exhausted (time beyond the last record)");
          break;
        }
        tc = tcn;
        t = t + h->cfg.dt;
      }
      chunk = s;
      p.series = h->series; p.nsite = h->nsite; p.nrec = h->nrec;
      p.win_first = first;
      p.win_len = tc - first + 1;
      if (p.win_len < 1) p.win_len = 1;
      if (p.win_first + p.win_len - 1 > h->nrec) p.win_len = h->nrec - p.win_first + 1;
      p.site_of_col = h->site_of_col; p.fscale = h->fscale; p.foffset = h->foffset;
    }
    if (need_lab) {
      // Records FLOOR(1 + time/dt) of every step a column runs in the chunk must exist in its set.  The device
      // accumulates time by repeated `+ dt`, which for a dt that is not exactly representable can sit an ulp above
      // k*dt: the bound is found by replaying the same additions, never by a multiplication.  Only the tail of a
      // series needs the replay.  A set whose columns have all passed their end step is not read any more.
      const double per_rec = tc8 ? 60.0 : h->cfg.dt;       // seconds per record
      const double t_last = tc8 ? 475200.0 : 1e300;          // the series is not read from this time on
      auto rec_at = [&](double t) { return (t < t_last) ? (long long)floor(1 + t / per_rec) : 1LL; };
      const long long first_rec = rec_at(h->time);
      for (size_t s = 0; s < h->lab_len.size(); s++) {
        if (h->lab_end[s] <= h->i) continue;
        const long long len = h->lab_len[s];
        const int64_t need = std::min<int64_t>(chunk, h->lab_end[s] - h->i);  // steps the set's columns run
        if (first_rec < 1 || first_rec > len) return fail(SAMSIM_ERR_STATE, "step: lab series exhausted");
        if (first_rec + (long long)((double)need * h->cfg.dt / per_rec) + 2 > len) {
          double t = h->time;
          int64_t ok = 0;
          for (; ok < need; ok++) {
            const long long rec = rec_at(t);
            if (rec < 1 || rec > len) break;
            t = t + h->cfg.dt;
          }
          if (ok < 1) return fail(SAMSIM_ERR_STATE, "step: lab series exhausted");
          if (ok < need) chunk = ok;
        }
      }
      p.lab = h->lab; p.lab_nrec = h->lab_nrec; p.set_of_col = h->set_of_col;
    }
    p.end_of_col = h->end_of_col;
    p.nsteps = (int)chunk;
    p.divergence = h->divergence;
    p.snap_sc = (h->snap_mode >= SAMSIM_SNAP_SCALARS) ? h->snap_sc : nullptr;
    p.snap_arr = (h->snap_mode >= SAMSIM_SNAP_FULL) ? h->snap_arr : nullptr;
    // small batches: shrink the block (the kernel is compiled for <= SAMSIM_BLOCK threads) until every SM has work
    int block = SAMSIM_BLOCK;
    while (block > 32 && (h->ncol + block - 1) / block < 4 * h->num_sms) block >>= 1;  // down to one warp per block: one warp per SM sub-partition
    const unsigned grid = (unsigned)((h->ncol + block - 1) / block);
    {
      int rc = claim_device_cfg(h);
      if (rc) return rc;
    }
    if (h->dcfg.two_pass) samsim_step_kernel<true><<<grid, block, 0, h->stream>>>(p);
    else samsim_step_kernel<false><<<grid, block, 0, h->stream>>>(p);
    CU(cudaGetLastError());
    CU(cudaEventRecord(h->ev_launch, h->stream));
    h->launches++;
    bool out = false;
    double out_time = 0.0;
    for (int64_t s = 0; s < chunk; s++) {
      out_time = h->time;
      out = clock_tick(h);
    }
    if (out && h->gs_ngroup > 0) {
      int rc = gs_record(h, out_time);
      if (rc) return rc;
    }
    if (out && h->ts_Q > 0) {
      int rc = ts_record(h, out_time);
      if (rc) return rc;
    }
    left -= chunk;
    if (h->rebin_every > 0 && (h->since_rebin += chunk) >= h->rebin_every) {
      h->since_rebin = 0;
      int rc = samsim_b200_rebin(h, nullptr);
      if (rc) return rc;
    }
  }
  CU(cudaEventRecord(h->ev1, h->stream));
  h->timed = true;
  // the last launch's divergence counters travel to pinned host memory behind the kernel; nobody waits for them here
  CU(cudaMemcpyAsync(h->divergence_host, h->divergence, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaEventRecord(h->ev_div, h->stream));
  h->div_pending = true;
  return 0;
}

// Re-bin the columns by regime (SURVEY 8e).  A warp costs as much as its deepest column and pays for every branch
// any of its lanes takes, so an ensemble whose columns have drifted apart (freeze-up at different dates, different
// snow states) runs faster once equal columns sit next to each other.  Columns are independent, so the order is
// free: a stable radix sort on (failed or finished, N_active, snow class, forcing site) gives the new order, every per-column
// row is permuted on the device, and slot_of_col / col_of_slot keep the caller's column numbering intact.
int samsim_b200_rebin(samsim_handle_t h, int32_t* changed) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (changed) *changed = 0;
  CU(cudaSetDevice(h->device));
  const long long n = h->ncol;
  const unsigned nb = (unsigned)((n + 255) / 256);
  unsigned long long *keys = nullptr, *keys_out = nullptr;
  int *vals = nullptr, *order = nullptr, *flag = nullptr;
  void *cub_tmp = nullptr, *tmp = nullptr;
  int rc = 0;
  auto cleanup = [&]() {
    cudaFree(keys); cudaFree(keys_out); cudaFree(vals); cudaFree(order); cudaFree(flag); cudaFree(cub_tmp); cudaFree(tmp);
  };
#define RB(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) { cleanup(); return fail(SAMSIM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } \
  } while (0)
  RB(cudaMalloc(&keys, (size_t)n * sizeof(unsigned long long)));
  RB(cudaMalloc(&keys_out, (size_t)n * sizeof(unsigned long long)));
  RB(cudaMalloc(&vals, (size_t)n * sizeof(int)));
  RB(cudaMalloc(&order, (size_t)n * sizeof(int)));
  RB(cudaMalloc(&flag, sizeof(int)));
  RB(cudaMemsetAsync(flag, 0, sizeof(int), h->stream));
  int site_bits = 0;  // bits of the largest site index
  while (h->site_of_col && (1ll << site_bits) < h->nsite) site_bits++;
  const int end_bit = 26 + site_bits;
  samsim_rebin_key_kernel<<<nb, 256, 0, h->stream>>>(h->sc, h->in, h->site_of_col, h->end_of_col, h->i, n, h->ncol_pad, h->cfg.thick_min,
                                                      site_bits, keys, vals);
  samsim_rebin_unsorted_kernel<<<nb, 256, 0, h->stream>>>(keys, n, flag);
  RB(cudaGetLastError());
  int unsorted = 0;
  RB(cudaMemcpyAsync(&unsorted, flag, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  RB(cudaStreamSynchronize(h->stream));
  if (unsorted == 0) { cleanup(); return 0; }  // already in regime order

  size_t cub_bytes = 0;
  RB(cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, keys, keys_out, vals, order, (int)n, 0, end_bit, h->stream));
  RB(cudaMalloc(&cub_tmp, cub_bytes));
  RB(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, keys, keys_out, vals, order, (int)n, 0, end_bit, h->stream));
  RB(cudaMalloc(&tmp, permute_tmp_bytes(h)));

  const size_t astr = (size_t)h->LS * h->ncol_pad;  // one array of the (row-major) snapshot buffer
  {
    // state arrays: gather array a of the columns in their new order into rows, write the rows back into the tiles
    const long long total = (long long)h->LS * n;
    const unsigned nbk = (unsigned)((total + 255) / 256);
    for (int a = 0; a < h->n_arr; a++) {
      if (a >= AR_STATE_COUNT && !(a >= AR_BGC1 && a < AR_BGC1 + h->cfg.N_bgc)) continue;  // scratch arrays carry no state
      samsim_state_to_rows_kernel<<<nbk, 256, 0, h->stream>>>(h->arr, (double*)tmp, n, h->ncol_pad, h->LS, h->n_arr, a, order);
      samsim_rows_to_state_kernel<<<nbk, 256, 0, h->stream>>>(h->arr, (const double*)tmp, n, h->ncol_pad, h->LS, h->n_arr, a);
    }
    RB(cudaGetLastError());
  }
  if (!rc) rc = permute_rows<double>(h, h->sc, SC_COUNT, order, tmp);
  if (!rc) rc = permute_rows<int>(h, h->in, IN_COUNT, order, tmp);
  if (!rc) rc = permute_rows<int>(h, h->site_of_col, 1, order, tmp);
  if (!rc) rc = permute_rows<int>(h, h->set_of_col, 1, order, tmp);
  if (!rc) rc = permute_rows<int64_t>(h, h->end_of_col, 1, order, tmp);
  if (!rc) rc = permute_rows<double>(h, h->fscale, 4, order, tmp);
  if (!rc) rc = permute_rows<double>(h, h->foffset, 4, order, tmp);
  if (!rc) rc = permute_rows<double>(h, h->snap_sc, SAMSIM_SNAPSC_COUNT, order, tmp);
  for (int a = 0; a < SAMSIM_SNAPARR_COUNT && !rc && h->snap_arr; a++) rc = permute_rows<double>(h, h->snap_arr + (size_t)a * astr, h->LS, order, tmp);
  if (rc) { cleanup(); return rc; }

  if (!h->slot_of_col) {
    RB(cudaMalloc(&h->slot_of_col, (size_t)n * sizeof(int)));
    // col_of_slot stays nullptr (= identity) for the maps kernel of the first re-binning
  }
  samsim_rebin_maps_kernel<<<nb, 256, 0, h->stream>>>(order, h->col_of_slot, (int*)tmp, h->slot_of_col, n);
  RB(cudaGetLastError());
  if (!h->col_of_slot) RB(cudaMalloc(&h->col_of_slot, (size_t)n * sizeof(int)));
  RB(cudaMemcpyAsync(h->col_of_slot, tmp, (size_t)n * sizeof(int), cudaMemcpyDeviceToDevice, h->stream));
  RB(cudaStreamSynchronize(h->stream));
#undef RB
  cleanup();
  h->rebins++;
  if (changed) *changed = 1;
  return 0;
}

int samsim_b200_set_tuning(samsim_handle_t h, int32_t two_pass, int32_t prefetch_layers) {
  if (!h || two_pass < 0 || two_pass > 1 || prefetch_layers < 0 || prefetch_layers > 64) return fail(SAMSIM_ERR_ARG, "set_tuning: bad argument");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  h->dcfg.two_pass = two_pass;
  if (prefetch_layers > 0) h->dcfg.pf = prefetch_layers;
  release_device_cfg(h);  // the next launch uploads the configuration again
  return 0;
}

int samsim_b200_set_rebin_interval(samsim_handle_t h, int64_t nsteps) {
  if (!h || nsteps < 0) return fail(SAMSIM_ERR_ARG, "set_rebin_interval: bad argument");
  h->rebin_every = nsteps;
  h->since_rebin = 0;
  return 0;
}

int samsim_b200_get_slot_map(samsim_handle_t h, int32_t* slot_of_col) {
  if (!h || !slot_of_col) return fail(SAMSIM_ERR_ARG, "get_slot_map: bad argument");
  CU(cudaSetDevice(h->device));
  if (!h->slot_of_col) {
    for (long long c = 0; c < h->ncol; c++) slot_of_col[c] = (int32_t)c;
    return 0;
  }
  CU(cudaMemcpyAsync(slot_of_col, h->slot_of_col, (size_t)h->ncol * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

// ---- binary checkpoint / restart (SURVEY 8f-4; the reference can only start from init) ----------------------
// File: "SAMB2CK1", sizeof(samsim_config_t), the config, ncol, the clock, then in the caller's column order
// arrays[id][col][extent], scalars[id][col], ints[id][col].  Forcing tables, end steps and lab lengths are run inputs,
// not state: set them again.
static const char CK_MAGIC[8] = {'S', 'A', 'M', 'B', '2', 'C', 'K', '2'};

int samsim_b200_save_checkpoint(samsim_handle_t h, const char* path) {
  if (!h || !path) return fail(SAMSIM_ERR_ARG, "save_checkpoint: bad argument");
  FILE* f = fopen(path, "wb");
  if (!f) return fail(SAMSIM_ERR_STATE, std::string("save_checkpoint: cannot open ") + path);
  const int64_t cfg_size = (int64_t)sizeof(samsim_config_t), ncol = h->ncol;
  const int64_t clock_i[3] = {h->i, h->n_time_out, h->time_counter};
  bool ok = fwrite(CK_MAGIC, 1, 8, f) == 8 && fwrite(&cfg_size, 8, 1, f) == 1 && fwrite(&h->cfg, sizeof h->cfg, 1, f) == 1 &&
            fwrite(&ncol, 8, 1, f) == 1 && fwrite(&h->time, 8, 1, f) == 1 && fwrite(clock_i, 8, 3, f) == 3;
  int rc = 0;
  const int32_t chunk = 65536;
  std::vector<double> buf;
  for (int id = 0; ok && !rc && id < SAMSIM_ARR_COUNT; id++) {
    const int ext = samsim_b200_array_extent(h, id);
    if (ext < 0) continue;  // tracer arrays of a run without tracers
    buf.resize((size_t)chunk * ext);
    for (int64_t c0 = 0; ok && !rc && c0 < ncol; c0 += chunk) {
      const int32_t n = (int32_t)((ncol - c0 < chunk) ? ncol - c0 : chunk);
      rc = samsim_b200_get_array(h, id, buf.data(), (int32_t)c0, n);
      if (!rc) ok = fwrite(buf.data(), sizeof(double), (size_t)n * ext, f) == (size_t)n * ext;
    }
  }
  buf.resize((size_t)ncol);
  for (int id = 0; ok && !rc && id < SAMSIM_SC_COUNT; id++) {
    rc = samsim_b200_get_scalar(h, id, buf.data(), 0, (int32_t)ncol);
    if (!rc) ok = fwrite(buf.data(), sizeof(double), (size_t)ncol, f) == (size_t)ncol;
  }
  std::vector<int32_t> ibuf((size_t)ncol);
  for (int id = 0; ok && !rc && id < SAMSIM_INT_COUNT; id++) {
    rc = samsim_b200_get_int(h, id, ibuf.data(), 0, (int32_t)ncol);
    if (!rc) ok = fwrite(ibuf.data(), sizeof(int32_t), (size_t)ncol, f) == (size_t)ncol;
  }
  ok = (fclose(f) == 0) && ok;
  if (rc) return rc;
  if (!ok) return fail(SAMSIM_ERR_STATE, std::string("save_checkpoint: short write to ") + path);
  return 0;
}

int samsim_b200_load_checkpoint(samsim_handle_t h, const char* path) {
  if (!h || !path) return fail(SAMSIM_ERR_ARG, "load_checkpoint: bad argument");
  FILE* f = fopen(path, "rb");
  if (!f) return fail(SAMSIM_ERR_STATE, std::string("load_checkpoint: cannot open ") + path);
  char magic[8];
  int64_t cfg_size = 0, ncol = 0, clock_i[3];
  samsim_config_t cfg;
  double time = 0.0;
  bool ok = fread(magic, 1, 8, f) == 8 && memcmp(magic, CK_MAGIC, 8) == 0 && fread(&cfg_size, 8, 1, f) == 1 &&
            cfg_size == (int64_t)sizeof(samsim_config_t) && fread(&cfg, sizeof cfg, 1, f) == 1 && fread(&ncol, 8, 1, f) == 1 &&
            fread(&time, 8, 1, f) == 1 && fread(clock_i, 8, 3, f) == 3;
  if (!ok) { fclose(f); return fail(SAMSIM_ERR_STATE, "load_checkpoint: not a samsim_b200 checkpoint of this version"); }
  if (ncol != h->ncol || memcmp(&cfg, &h->cfg, sizeof cfg) != 0) {
    fclose(f);
    return fail(SAMSIM_ERR_CONFIG, "load_checkpoint: the handle was created with another configuration or column count");
  }
  int rc = 0;
  const int32_t chunk = 65536;
  std::vector<double> buf;
  for (int id = 0; ok && !rc && id < SAMSIM_ARR_COUNT; id++) {
    const int ext = samsim_b200_array_extent(h, id);
    if (ext < 0) continue;
    buf.resize((size_t)chunk * ext);
    for (int64_t c0 = 0; ok && !rc && c0 < ncol; c0 += chunk) {
      const int32_t n = (int32_t)((ncol - c0 < chunk) ? ncol - c0 : chunk);
      ok = fread(buf.data(), sizeof(double), (size_t)n * ext, f) == (size_t)n * ext;
      if (ok) rc = samsim_b200_set_array(h, id, buf.data(), (int32_t)c0, n);
    }
  }
  buf.resize((size_t)ncol);
  for (int id = 0; ok && !rc && id < SAMSIM_SC_COUNT; id++) {
    ok = fread(buf.data(), sizeof(double), (size_t)ncol, f) == (size_t)ncol;
    if (ok) rc = samsim_b200_set_scalar(h, id, buf.data(), 0, (int32_t)ncol);
  }
  std::vector<int32_t> ibuf((size_t)ncol);
  for (int id = 0; ok && !rc && id < SAMSIM_INT_COUNT; id++) {
    ok = fread(ibuf.data(), sizeof(int32_t), (size_t)ncol, f) == (size_t)ncol;
    if (ok) rc = samsim_b200_set_int(h, id, ibuf.data(), 0, (int32_t)ncol);
  }
  fclose(f);
  if (rc) return rc;
  if (!ok) return fail(SAMSIM_ERR_STATE, "load_checkpoint: truncated file");
  h->time = time; h->i = clock_i[0]; h->n_time_out = (int)clock_i[1]; h->time_counter = (int)clock_i[2];
  return 0;
}

int samsim_b200_synchronize(samsim_handle_t h) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int samsim_b200_set_snapshot_mode(samsim_handle_t h, int32_t mode) {
  if (!h || mode < 0 || mode > 2) return fail(SAMSIM_ERR_ARG, "set_snapshot_mode: bad argument");
  if (h->gs_ngroup > 0 && mode < (h->gs_mask ? SAMSIM_SNAP_FULL : SAMSIM_SNAP_SCALARS))
    return fail(SAMSIM_ERR_STATE, "set_snapshot_mode: the group statistics read this snapshot (switch them off first)");
  if (h->ts_Q > 0 && mode < (h->ts_mask ? SAMSIM_SNAP_FULL : SAMSIM_SNAP_SCALARS))
    return fail(SAMSIM_ERR_STATE, "set_snapshot_mode: the time statistics read this snapshot (switch them off first)");
  CU(cudaSetDevice(h->device));
  if (mode >= SAMSIM_SNAP_SCALARS && !h->snap_sc) {
    CU(cudaMalloc(&h->snap_sc, (size_t)SAMSIM_SNAPSC_COUNT * h->ncol_pad * sizeof(double)));
    CU(cudaMemset(h->snap_sc, 0, (size_t)SAMSIM_SNAPSC_COUNT * h->ncol_pad * sizeof(double)));
  }
  if (mode >= SAMSIM_SNAP_FULL && !h->snap_arr) {
    const size_t nb = (size_t)SAMSIM_SNAPARR_COUNT * h->LS * h->ncol_pad * sizeof(double);
    CU(cudaMalloc(&h->snap_arr, nb));
    CU(cudaMemset(h->snap_arr, 0, nb));
  }
  h->snap_mode = mode;
  return 0;
}

int samsim_b200_get_snapshot(samsim_handle_t h, double* scalars, double* arrays, int32_t col0, int32_t n) {
  int rc = check_cols(h, col0, n);
  if (rc) return rc;
  if (h->snap_mode == SAMSIM_SNAP_NONE) return fail(SAMSIM_ERR_STATE, "get_snapshot: snapshot mode is NONE");
  if (arrays && h->snap_mode < SAMSIM_SNAP_FULL) return fail(SAMSIM_ERR_STATE, "get_snapshot: arrays need SAMSIM_SNAP_FULL");
  if (n == 0) return 0;
  CU(cudaSetDevice(h->device));
  if (scalars) {
    const size_t bytes = (size_t)n * SAMSIM_SNAPSC_COUNT * sizeof(double);
    if ((rc = ensure_stage(h, bytes))) return rc;
    const long long total = (long long)n * SAMSIM_SNAPSC_COUNT;
    // scalars are [id][ncol_pad]: treat as count=SNAPSC_COUNT arrays of extent 1 with LS=1
    samsim_gather_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(h->snap_sc, h->stage, h->ncol_pad, 1, SAMSIM_SNAPSC_COUNT, 1, col0, n, 0, h->slot_of_col);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(scalars, h->stage, bytes, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  if (arrays) {
    const int ext = h->cfg.Nlayer;
    const size_t bytes = (size_t)n * SAMSIM_SNAPARR_COUNT * ext * sizeof(double);
    if ((rc = ensure_stage(h, bytes))) return rc;
    const long long total = (long long)n * SAMSIM_SNAPARR_COUNT * ext;
    samsim_gather_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(h->snap_arr, h->stage, h->ncol_pad, h->LS, SAMSIM_SNAPARR_COUNT, ext, col0, n, 1, h->slot_of_col);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(arrays, h->stage, bytes, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  return 0;
}

// The depth grid and profiles of the group and time statistics, and the snapshot they need (SAMSIM_ERR_ARG /
// SAMSIM_ERR_STATE with the caller's name)
static int check_depth_grid(samsim_handle_t h, int32_t nz, const double* depth, uint32_t profile_mask, const char* who) {
  const std::string w = std::string(who) + ": ";
  if (nz < 0 || (nz > 0 && !depth)) return fail(SAMSIM_ERR_ARG, w + "bad depth grid");
  for (int32_t j = 0; j < nz; j++)
    if (!isfinite(depth[j]) || !(depth[j] > 0.0) || (j > 0 && !(depth[j] > depth[j - 1])))
      return fail(SAMSIM_ERR_ARG, w + "depths must be finite, > 0 and strictly increasing");
  if (profile_mask >> SAMSIM_SNAPARR_COUNT) return fail(SAMSIM_ERR_ARG, w + "unknown snapshot array in profile_mask");
  if (profile_mask & (1u << SAMSIM_SNAPARR_RAY))
    return fail(SAMSIM_ERR_ARG, w + "ray is an interface quantity (extent Nlayer-1), not a layer profile");
  for (int a = SAMSIM_SNAPARR_BGC1_BU; a < SAMSIM_SNAPARR_COUNT; a++)
    if ((profile_mask >> a & 1u) && (a - SAMSIM_SNAPARR_BGC1_BU) / 2 >= h->cfg.N_bgc)
      return fail(SAMSIM_ERR_ARG, w + "tracer rows need N_bgc tracers");
  if (profile_mask && nz == 0) return fail(SAMSIM_ERR_ARG, w + "profiles need a depth grid (nz > 0)");
  if (h->snap_mode < (profile_mask ? SAMSIM_SNAP_FULL : SAMSIM_SNAP_SCALARS))
    return fail(SAMSIM_ERR_STATE, w + "needs snapshot mode SCALARS, or FULL for profiles");
  return 0;
}

int samsim_b200_set_group_stats(samsim_handle_t h, int32_t ngroup, const int32_t* group_of_col, int32_t nz,
                                const double* depth, uint32_t profile_mask, int32_t max_records) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (ngroup == 0) {  // off
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    gs_free(h);
    return 0;
  }
  // every argument is checked before the previous setting is dropped
  if (ngroup < 0 || ngroup >= (1 << 26)) return fail(SAMSIM_ERR_ARG, "set_group_stats: ngroup must be in 0 .. 2^26-1");
  if (max_records < 1) return fail(SAMSIM_ERR_ARG, "set_group_stats: max_records must be >= 1");
  if (group_of_col)
    for (long long c = 0; c < h->ncol; c++)
      if (group_of_col[c] < -1 || group_of_col[c] >= ngroup) return fail(SAMSIM_ERR_ARG, "set_group_stats: group index out of [-1, ngroup)");
  {
    int rc = check_depth_grid(h, nz, depth, profile_mask, "set_group_stats");
    if (rc) return rc;
  }
  int nprof = 0;
  int prof[SAMSIM_SNAPARR_COUNT];
  for (int a = 0; a < SAMSIM_SNAPARR_COUNT; a++)
    if (profile_mask >> a & 1u) prof[nprof++] = a;
  const int Q = SAMSIM_GS_NSC + nprof * nz;
  const GsLayout L = gs_layout(h->ncol, ngroup, group_of_col);
  std::vector<int32_t> big;  // [3][nbig]: group, first tile, log2 size
  for (int32_t g = 0; g < ngroup; g++)
    if (L.lg[(size_t)g] > 10) big.push_back(g);
  const int nbig = (int)big.size();
  big.resize(3 * (size_t)nbig);
  for (int b = 0; b < nbig; b++) {
    big[(size_t)nbig + b] = (int32_t)(L.start[(size_t)big[b]] / SAMSIM_GS_TILE);
    big[2 * (size_t)nbig + b] = L.lg[(size_t)big[b]];
  }

  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  gs_free(h);
  const size_t np = (size_t)L.npad, npart = (size_t)Q * (np / SAMSIM_GS_TILE);
  const size_t nhist = (size_t)max_records * ngroup * Q * 5;
  cudaError_t e;
  if ((e = cudaMalloc(&h->gs_col, np * sizeof(int))) != cudaSuccess || (e = cudaMalloc(&h->gs_info, np * sizeof(int))) != cudaSuccess ||
      (e = cudaMalloc(&h->gs_big, (big.size() + 1) * sizeof(int))) != cudaSuccess ||
      (e = cudaMalloc(&h->gs_z, ((size_t)nz + 1) * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->gs_vals, (size_t)Q * np * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->gs_reach, np * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->gs_part, 4 * npart * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->gs_hist, nhist * sizeof(double))) != cudaSuccess ||
      (e = cudaMemcpy(h->gs_col, L.col.data(), np * sizeof(int), cudaMemcpyHostToDevice)) != cudaSuccess ||
      (e = cudaMemcpy(h->gs_info, L.info.data(), np * sizeof(int), cudaMemcpyHostToDevice)) != cudaSuccess ||
      (nbig && (e = cudaMemcpy(h->gs_big, big.data(), big.size() * sizeof(int), cudaMemcpyHostToDevice)) != cudaSuccess) ||
      (nz && (e = cudaMemcpy(h->gs_z, depth, (size_t)nz * sizeof(double), cudaMemcpyHostToDevice)) != cudaSuccess)) {
    gs_free(h);
    cudaGetLastError();
    return fail(SAMSIM_ERR_CUDA, std::string("set_group_stats: ") + cudaGetErrorString(e));
  }
  h->gs_ngroup = ngroup; h->gs_Q = Q; h->gs_nz = nz; h->gs_nprof = nprof; h->gs_max = max_records; h->gs_held = 0;
  for (int a = 0; a < nprof; a++) h->gs_prof[a] = prof[a];
  h->gs_mask = profile_mask; h->gs_npad = L.npad; h->gs_nbig = nbig;
  h->gs_time.assign((size_t)max_records, 0.0);
  h->gs_i.assign((size_t)max_records, 0);
  return 0;
}

int32_t samsim_b200_group_stats_held(samsim_handle_t h) { return h ? h->gs_held : -1; }

int samsim_b200_get_group_stats(samsim_handle_t h, double* stats, double* rec_time, int64_t* rec_i, int32_t rec0, int32_t nrec) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (rec0 < 0 || nrec < 0 || (int64_t)rec0 + nrec > h->gs_held)
    return fail(SAMSIM_ERR_ARG, "get_group_stats: records rec0 .. rec0+nrec-1 must be held");
  if (nrec == 0) return 0;
  if (rec_time) std::copy(h->gs_time.begin() + rec0, h->gs_time.begin() + rec0 + nrec, rec_time);
  if (rec_i) std::copy(h->gs_i.begin() + rec0, h->gs_i.begin() + rec0 + nrec, rec_i);
  if (stats) {
    CU(cudaSetDevice(h->device));
    const size_t per = (size_t)h->gs_ngroup * h->gs_Q * 5;
    CU(cudaMemcpyAsync(stats, h->gs_hist + (size_t)rec0 * per, (size_t)nrec * per * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  return 0;
}

int samsim_b200_clear_group_stats(samsim_handle_t h) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  h->gs_held = 0;
  return 0;
}

int samsim_b200_set_time_stats(samsim_handle_t h, int32_t records_per_window, uint32_t scalar_mask, int32_t nz,
                               const double* depth, uint32_t profile_mask, int32_t max_windows) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (scalar_mask == 0 && profile_mask == 0) {  // off
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    ts_free(h);
    return 0;
  }
  // every argument is checked before the previous setting is dropped
  if (records_per_window < 0) return fail(SAMSIM_ERR_ARG, "set_time_stats: records_per_window must be >= 0");
  if (max_windows < 1) return fail(SAMSIM_ERR_ARG, "set_time_stats: max_windows must be >= 1");
  if (scalar_mask >> SAMSIM_SNAPSC_COUNT) return fail(SAMSIM_ERR_ARG, "set_time_stats: unknown snapshot scalar in scalar_mask");
  {
    int rc = check_depth_grid(h, nz, depth, profile_mask, "set_time_stats");
    if (rc) return rc;
  }
  int nsc = 0, nprof = 0;
  int sc[SAMSIM_SNAPSC_COUNT], prof[SAMSIM_SNAPARR_COUNT];
  for (int q = 0; q < SAMSIM_SNAPSC_COUNT; q++)
    if (scalar_mask >> q & 1u) sc[nsc++] = q;
  for (int a = 0; a < SAMSIM_SNAPARR_COUNT; a++)
    if (profile_mask >> a & 1u) prof[nprof++] = a;
  const int Q = nsc + nprof * (profile_mask ? nz : 0);

  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  ts_free(h);
  const size_t per = (size_t)Q * SAMSIM_TS_NSTAT * h->ncol_pad;  // doubles of one window
  cudaError_t e;
  if ((e = cudaMalloc(&h->ts_z, ((size_t)nz + 1) * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->ts_acc, per * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->ts_hist, (size_t)max_windows * per * sizeof(double))) != cudaSuccess ||
      (nz && (e = cudaMemcpy(h->ts_z, depth, (size_t)nz * sizeof(double), cudaMemcpyHostToDevice)) != cudaSuccess)) {
    ts_free(h);
    cudaGetLastError();
    return fail(SAMSIM_ERR_CUDA, std::string("set_time_stats: ") + cudaGetErrorString(e));
  }
  h->ts_Q = Q; h->ts_nsc = nsc; h->ts_nz = profile_mask ? nz : 0; h->ts_nprof = nprof;
  h->ts_rpw = records_per_window; h->ts_max = max_windows; h->ts_held = 0; h->ts_cur = 0;
  for (int q = 0; q < nsc; q++) h->ts_sc[q] = sc[q];
  for (int a = 0; a < nprof; a++) h->ts_prof[a] = prof[a];
  h->ts_mask = profile_mask;
  h->ts_nrec.assign((size_t)max_windows, 0);
  h->ts_time.assign(2 * ((size_t)max_windows + 1), 0.0);
  h->ts_i.assign(2 * ((size_t)max_windows + 1), 0);
  return 0;
}

int32_t samsim_b200_time_stats_held(samsim_handle_t h) { return h ? h->ts_held : -1; }

int samsim_b200_get_time_stats(samsim_handle_t h, double* stats, int32_t* win_nrec, double* win_time, int64_t* win_i,
                               int32_t win0, int32_t nwin, int32_t col0, int32_t n) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (win0 < 0 || nwin < 0 || (int64_t)win0 + nwin > h->ts_held)
    return fail(SAMSIM_ERR_ARG, "get_time_stats: windows win0 .. win0+nwin-1 must be held");
  if (col0 < 0 || n < 0 || (int64_t)col0 + n > h->ncol) return fail(SAMSIM_ERR_ARG, "get_time_stats: column range out of bounds");
  if (nwin == 0) return 0;
  if (win_nrec) std::copy(h->ts_nrec.begin() + win0, h->ts_nrec.begin() + win0 + nwin, win_nrec);
  if (win_time) std::copy(h->ts_time.begin() + 2 * (size_t)win0, h->ts_time.begin() + 2 * ((size_t)win0 + nwin), win_time);
  if (win_i) std::copy(h->ts_i.begin() + 2 * (size_t)win0, h->ts_i.begin() + 2 * ((size_t)win0 + nwin), win_i);
  if (stats && n > 0) {
    CU(cudaSetDevice(h->device));
    const size_t per_col = (size_t)h->ts_Q * SAMSIM_TS_NSTAT, per_win = per_col * h->ncol_pad;
    // staged in pieces of at most 2^25 doubles (256 MB)
    const int64_t cols = std::max<int64_t>(1, std::min<int64_t>(n, ((int64_t)1 << 25) / (int64_t)per_col));
    int rc;
    if ((rc = ensure_stage(h, (size_t)cols * per_col * sizeof(double)))) return rc;
    for (int32_t w = 0; w < nwin; w++)
      for (int64_t c0 = 0; c0 < n; c0 += cols) {
        const int64_t m = std::min<int64_t>(cols, n - c0);
        const long long total = m * (long long)per_col;
        samsim_ts_get_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(
            h->ts_hist + (size_t)(win0 + w) * per_win, h->stage, h->ncol_pad, h->ts_Q, col0 + c0, m);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(stats + ((size_t)w * n + c0) * per_col, h->stage, (size_t)total * sizeof(double),
                           cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
      }
  }
  return 0;
}

int samsim_b200_close_time_window(samsim_handle_t h) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (h->ts_Q == 0) return fail(SAMSIM_ERR_STATE, "close_time_window: time statistics are off");
  if (h->ts_cur == 0) return fail(SAMSIM_ERR_STATE, "close_time_window: the window in progress holds no record");
  if (h->ts_held >= h->ts_max)
    return fail(SAMSIM_ERR_STATE, "close_time_window: the history is full (samsim_b200_get_time_stats / _clear_time_stats)");
  CU(cudaSetDevice(h->device));
  samsim_ts_close_kernel<<<(unsigned)((h->ncol + 255) / 256), 256, 0, h->stream>>>(
      h->ts_acc, h->ts_hist + (size_t)h->ts_held * h->ts_Q * SAMSIM_TS_NSTAT * h->ncol_pad, h->ts_Q, h->ncol, h->ncol_pad);
  CU(cudaGetLastError());
  ts_window_done(h);
  return 0;
}

int samsim_b200_clear_time_stats(samsim_handle_t h) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  h->ts_held = 0;
  return 0;
}

int samsim_b200_get_status(samsim_handle_t h, int32_t* status, int32_t col0, int32_t n) {
  return samsim_b200_get_int(h, SAMSIM_INT_STATUS, status, col0, n);
}

int samsim_b200_count_failed(samsim_handle_t h, int32_t* nfailed) {
  if (!h || !nfailed) return fail(SAMSIM_ERR_ARG, "count_failed: bad argument");
  CU(cudaSetDevice(h->device));
  int rc;
  if ((rc = ensure_stage(h, sizeof(int)))) return rc;
  CU(cudaMemsetAsync(h->stage, 0, sizeof(int), h->stream));
  samsim_count_failed_kernel<<<(unsigned)((h->ncol + 255) / 256), 256, 0, h->stream>>>(h->in, h->ncol, h->ncol_pad, (int*)h->stage);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(nfailed, h->stage, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return 0;
}

int samsim_b200_reduce_diag(samsim_handle_t h, double* out18) {
  if (!h || !out18) return fail(SAMSIM_ERR_ARG, "reduce_diag: bad argument");
  CU(cudaSetDevice(h->device));
  const unsigned nb = (unsigned)((h->ncol + 127) / 128);
  int rc;
  if ((rc = ensure_stage(h, (size_t)nb * 18 * sizeof(double)))) return rc;
  samsim_reduce_kernel<<<nb, 128, 0, h->stream>>>(h->sc, h->in, h->ncol, h->ncol_pad, h->stage);
  CU(cudaGetLastError());
  std::vector<double> part((size_t)nb * 18);
  CU(cudaMemcpyAsync(part.data(), h->stage, part.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  for (int j = 0; j < 6; j++) {
    double s = 0.0, mn = 1e300, mx = -1e300;
    for (unsigned b = 0; b < nb; b++) {
      s += part[((size_t)b * 6 + j) * 3 + 0];
      mn = fmin(mn, part[((size_t)b * 6 + j) * 3 + 1]);
      mx = fmax(mx, part[((size_t)b * 6 + j) * 3 + 2]);
    }
    out18[3 * j + 0] = s; out18[3 * j + 1] = mn; out18[3 * j + 2] = mx;
  }
  return 0;
}

int64_t samsim_b200_launch_count(samsim_handle_t h) { return h ? h->launches : -1; }

int samsim_b200_last_step_ms(samsim_handle_t h, float* ms) {
  if (!h || !ms) return fail(SAMSIM_ERR_ARG, "last_step_ms: bad argument");
  if (!h->timed) return fail(SAMSIM_ERR_STATE, "last_step_ms: no step yet");
  CU(cudaSetDevice(h->device));
  CU(cudaEventSynchronize(h->ev1));
  CU(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  return 0;
}

int samsim_b200_device_layout(samsim_handle_t h, void** arrays, void** scalars, void** ints, int64_t* ncol_pad, int64_t* lstride,
                              int64_t* narrays) {
  if (!h) return fail(SAMSIM_ERR_ARG, "null handle");
  if (arrays) *arrays = h->arr;
  if (scalars) *scalars = h->sc;
  if (ints) *ints = h->in;
  if (ncol_pad) *ncol_pad = h->ncol_pad;
  if (lstride) *lstride = h->LS;
  if (narrays) *narrays = h->n_arr;
  return 0;
}

// ---- KATs -------------------------------------------------------------------------------------
static int kat_common(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return fail(SAMSIM_ERR_NO_DEVICE, "no CUDA device: samsim_b200 has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(SAMSIM_ERR_ARG, "bad device index");
  CU(cudaSetDevice(device));
  return 0;
}
// the known-answer kernels read the liquidus of `salt_flag` from the constant-memory configuration
static int kat_upload_cfg(int device, int salt_flag) {
  if (!(salt_flag == 1 || salt_flag == 2)) return fail(SAMSIM_ERR_ARG, "salt_flag must be 1 or 2");
  DevCfg g;
  memset(&g, 0, sizeof g);
  fill_liquidus(g, salt_flag);
  std::lock_guard<std::mutex> lock(g_cfg_mutex);
  CU(cudaDeviceSynchronize());  // no step kernel of another handle may still be reading the old configuration
  CU(cudaMemcpyToSymbol(samsim_dev_cfg, &g, sizeof(DevCfg), 0, cudaMemcpyHostToDevice));
  g_cfg_owner[device & 63] = nullptr;
  return 0;
}

int samsim_b200_kat_getT(int32_t salt_flag, int32_t n, const double* H, const double* S_bu, const double* T_in, double* T_out,
                         double* phi_out, int32_t* status_out, int32_t device) {
  int rc = kat_common(device);
  if (rc) return rc;
  if (n < 1 || !H || !S_bu || !T_in || !T_out || !phi_out) return fail(SAMSIM_ERR_ARG, "kat_getT: bad argument");
  if ((rc = kat_upload_cfg(device, salt_flag))) return rc;
  double* d = nullptr;
  int* ds = nullptr;
  const size_t nb = (size_t)n * sizeof(double);
  CU(cudaMalloc(&d, 5 * nb));
  CU(cudaMalloc(&ds, (size_t)n * sizeof(int)));
  CU(cudaMemcpy(d, H, nb, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(d + n, S_bu, nb, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(d + 2 * (size_t)n, T_in, nb, cudaMemcpyHostToDevice));
  samsim_kat_getT_kernel<<<(n + 127) / 128, 128>>>(salt_flag, n, d, d + n, d + 2 * (size_t)n, d + 3 * (size_t)n, d + 4 * (size_t)n, ds);
  CU(cudaGetLastError());
  CU(cudaMemcpy(T_out, d + 3 * (size_t)n, nb, cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(phi_out, d + 4 * (size_t)n, nb, cudaMemcpyDeviceToHost));
  if (status_out) CU(cudaMemcpy(status_out, ds, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost));
  cudaFree(d);
  cudaFree(ds);
  return 0;
}

int samsim_b200_kat_scalar(int32_t fn, int32_t salt_flag, int32_t n, const double* a, const double* b, double* out, int32_t device) {
  int rc = kat_common(device);
  if (rc) return rc;
  if (n < 1 || !a || !out) return fail(SAMSIM_ERR_ARG, "kat_scalar: bad argument");
  if ((rc = kat_upload_cfg(device, salt_flag))) return rc;
  double* d = nullptr;
  const size_t nb = (size_t)n * sizeof(double);
  CU(cudaMalloc(&d, 3 * nb));
  CU(cudaMemcpy(d, a, nb, cudaMemcpyHostToDevice));
  if (b) CU(cudaMemcpy(d + n, b, nb, cudaMemcpyHostToDevice));
  else CU(cudaMemset(d + n, 0, nb));
  samsim_kat_scalar_kernel<<<(n + 127) / 128, 128>>>(fn, salt_flag, n, d, d + n, d + 2 * (size_t)n);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, d + 2 * (size_t)n, nb, cudaMemcpyDeviceToHost));
  cudaFree(d);
  return 0;
}

int samsim_b200_fp64_peak(int32_t device, double seconds, double* tflops) {
  int rc = kat_common(device);
  if (rc) return rc;
  if (!tflops) return fail(SAMSIM_ERR_ARG, "fp64_peak: bad argument");
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256;
  double* d = nullptr;
  CU(cudaMalloc(&d, (size_t)blocks * threads * sizeof(double)));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  int iters = 2000;
  double best = 0.0, elapsed_total = 0.0;
  samsim_fp64_peak_kernel<<<blocks, threads>>>(d, 100, 1.0);  // warm-up
  CU(cudaDeviceSynchronize());
  while (elapsed_total < seconds * 1000.0) {
    cudaEventRecord(e0);
    samsim_fp64_peak_kernel<<<blocks, threads>>>(d, iters, 1.0);
    cudaEventRecord(e1);
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    elapsed_total += ms;
    const double flop = 2.0 * 64.0 * (double)iters * blocks * threads;  // 8 chains x 8 unroll fma = 64 fma/iter
    const double tf = flop / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
    if (ms < 50.f) iters *= 2;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *tflops = best;
  return 0;
}

}  // extern "C"
