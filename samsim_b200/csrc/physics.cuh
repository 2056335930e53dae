// physics.cuh -- per-column device physics of the SAMSIM timestep for sm_100a.
//
// One thread owns one column.  Per-layer arrays live in a warp-tiled SoA device buffer: the 32 columns of a warp
// form a tile, and element (array a, layer k) of column c is
//     arr[(((c/32)*LS + k)*NA + a)*32 + c%32]            LS = Nlayer+2, NA = number of arrays
// so that (1) the 32 columns of a warp touch 32 consecutive doubles (one 256-byte request) for every per-layer
// access, (2) all arrays of one layer sit next to each other: from the thread's layer pointer base + k*(NA*32) every
// array is a compile-time immediate offset a*256 B (no per-access address arithmetic: the first layout,
// [a][k][column], spent 30 % of the kernel's instructions on IMAD/LEA/UMOV/R2UR address computation), and (3) a
// warp's whole state is one contiguous 0.5 MB region (one TLB entry, DRAM pages shared by the arrays of a layer)
// instead of 2200 rows 8 MB apart.  Per-column scalars are loaded into the Col struct (registers / local memory)
// for the duration of a launch.
//
// Arithmetic contract: this file is compiled with -fmad=false; every expression keeps the
// reference's left-to-right operation order, the transcendental calls go through detmath.h,
// and x**2._wp / x**3._wp / x**4._wp are products.  Under that contract the results are
// bit-identical with the CPU oracle's "det" build (tests/test_parity_*.py).
//
// Each function cites the reference routine it replaces (paths relative to /root/reference).
#pragma once

#include <stdint.h>

#include "detmath.h"
#include "params.cuh"

namespace samsim {

// ---- run-wide configuration in constant memory -------------------------------------------
struct DevCfg {
  int testcase;
  int Nlayer, N_top, N_middle, N_bottom;
  int atmoflux_flag, grav_flag, prescribe_flag, grav_heat_flag, flush_heat_flag, turb_flag, salt_flag,
      boundflux_flag, flush_flag, flood_flag, bottom_flag, precip_flag, harmonic_flag, tank_flag, albedo_flag,
      lab_snow_flag, freeboard_snow_flag, snow_flush_flag, snow_precip_flag;
  int i_time_out;
  int n_bgc;  // 0: bgc_flag 1 (no tracers); 1..2: bgc_flag 2 with that many passive tracers
  double dt, thick_0, thick_min, time_out;
  double alpha_flux_instable, alpha_flux_stable, m_total;
  double max_flux_plate, k_snow_flush, k_styropor;
  // liquidus coefficients for salt_flag
  double c2, c3, c4, d2, d3x2, d4x3;
  // tuning (samsim_b200_set_tuning; results do not depend on it)
  int two_pass;   // 1: steady columns take the merged forward / backward passes of step.cuh
  int pf;         // L1 prefetch distance of the layer sweeps, in layers
};

// The configuration of the running launch.  On the device it lives in constant memory so that flags, dt and the
// liquidus coefficients are constant-bank operands of the arithmetic instructions (passed by reference through the
// call tree they were generic loads: three per liquidus evaluation).  samsim_b200_step uploads the handle's DevCfg
// before a launch whenever another handle used the device last.
#ifdef SAMSIM_HOST_BUILD
static const DevCfg* samsim_host_cfg = nullptr;   // tests/hostbuild: set by the harness before column_step
#define CFG (*samsim::samsim_host_cfg)
#else
__constant__ DevCfg samsim_dev_cfg;
#define CFG samsim::samsim_dev_cfg
#endif

// scalar slots: MUST stay in the order of samsim_scalar_id (include/samsim_b200.h)
enum {
  SC_T_BOTTOM = 0, SC_T_TOP, SC_S_BU_BOTTOM, SC_T2M, SC_FL_Q_BOTTOM,
  SC_PSI_S_SNOW, SC_PSI_L_SNOW, SC_PSI_G_SNOW, SC_PHI_S, SC_S_ABS_SNOW, SC_H_ABS_SNOW, SC_M_SNOW, SC_T_SNOW,
  SC_THICK_SNOW, SC_LIQUID_PRECIP, SC_SOLID_PRECIP, SC_FL_Q_SNOW,
  SC_ENERGY_STORED, SC_TOTAL_RESIST, SC_FRESHWATER, SC_THICKNESS, SC_BULK_SALIN,
  SC_ALBEDO, SC_FL_SW, SC_FL_LW, SC_FL_REST,
  SC_GRAV_DRAIN, SC_GRAV_SALT, SC_GRAV_TEMP,
  SC_MELT_THICK, SC_MELT_THICK_SNOW, SC_MELT_THICK_SNOW_OLD,
  SC_MTO1, SC_MTO2, SC_MTO3,
  SC_FREEBOARD, SC_T_FREEZE, SC_MELT_ERR, SC_S_TOTAL,
  SC_TTOP_WARM, SC_TTOP_COLD, SC_OFLUX_AMP,
  SC_BGC_BOTTOM1, SC_BGC_BOTTOM2, SC_BGC_TOTAL1, SC_BGC_TOTAL2,
  SC_COUNT
};
// array slots: first ARR_STATE_COUNT in the order of samsim_array_id, then launch-local scratch
enum {
  AR_M = 0, AR_S_ABS, AR_H_ABS, AR_THICK, AR_T, AR_PHI, AR_S_BU, AR_PSI_S, AR_PSI_L, AR_PSI_G, AR_RAY, AR_PERM,
  AR_FLUSH_V, AR_FLUSH_H, AR_FL_Q,
  AR_STATE_COUNT,
  AR_S_BR = AR_STATE_COUNT, AR_V_EX, AR_FL_M, AR_W0, AR_W1, AR_W2, AR_W3,
  AR_CORE_COUNT,
  // passive tracers (allocated only when n_bgc > 0): state bgc_abs(:,1:2), then the step-local sparse form of the
  // brine-flux matrix fl_brine_bgc (see fb_cell)
  AR_BGC1 = AR_CORE_COUNT, AR_BGC2, AR_FB_D, AR_FB_U, AR_FB_A, AR_FB_O,
  AR_COUNT
};
enum { IN_N_ACTIVE = 0, IN_STATUS, IN_STYROPOR, IN_EVENTS0, IN_EVENTS1, IN_COUNT };

// Branch events (samsim_event_id of include/samsim_b200.h, same order): bit id of the per-column event words is set
// when the column executes the branch.  They let a parity test prove that the branch it claims to cover ran; the
// CPU oracle counts the same branches.  Not part of the model state.
enum {
  EV_FLOOD = 0, EV_FLOOD_NEG_FREE, EV_FLOOD_SIMPLE, EV_FLUSH3, EV_FLUSH4, EV_FLUSH_INLINE, EV_STYROPOR, EV_SNOW_THERMO,
  EV_SNOW_THERMO_MELTWATER, EV_SNOW_WET, EV_SNOW_MERGE, EV_SNOW_COMPACTION, EV_SNOW_COUPLING_ITER,
  EV_SNOW_COUPLING_WARM1, EV_SNOW_COUPLING_WARM2, EV_SNOW_PRECIP, EV_SNOW_PRECIP_0, EV_MELT_SNOW_ALL, EV_MELT_SNOW_PART,
  EV_BOTTOM_MELT, EV_BOTTOM_MELT_SIMPLE_A, EV_BOTTOM_MELT_SIMPLE_B, EV_BOTTOM_GROWTH_SIMPLE, EV_BOTTOM_GROWTH,
  EV_TOP_GROW_A, EV_TOP_GROW_B, EV_TOP_GROW_C, EV_TOP_MELT_A, EV_TOP_MELT_B, EV_TOP_MELT_C, EV_GRAV_DRAINED,
  EV_SALT_CLAMP,
  EV_GAS_REFILL, EV_GETT_TFR_FALLBACK, EV_GETT_SALTFREE, EV_GETT_LIQUID, EV_HEAT_MELT, EV_HEAT_THIN_SNOW,
  EV_MELT_THICK_GAS, EV_SNOW_MELTWATER_TO_ICE, EV_PRESCRIBE, EV_GRAV_DRAIN_SIMPLE, EV_NOTZFLUX, EV_FLUSH3_CLAMP,
  EV_SCRUB, EV_MELT_THICK, EV_TURB, EV_TANK, EV_TWO_PASS_STEP,
  EV_COUNT
};

// strided per-layer view of one column (1-based layer index like the reference)
struct Lay {
  double* p;    // &arr[tile][0][a][lane]
  unsigned ls;  // NA*32: elements between consecutive layers of the tile (32-bit index arithmetic inside a tile)
  __device__ __forceinline__ double& operator[](int k) const {
#if !defined(SAMSIM_HOST_BUILD) && defined(__CUDA_ARCH__)
    __builtin_assume(__isGlobal(p));  // ld.global / st.global instead of generic accesses
#endif
    return p[(unsigned)k * ls];
  }
  // non-blocking L1 prefetch of layer k (sweeps are latency bound: one 256-byte warp request per layer and
  // array, no spatial reuse between layers); k is clamped by the callers to [0, Nlayer+1]
  __device__ __forceinline__ void prefetch(int k) const {
#ifndef SAMSIM_HOST_BUILD   // (tests/hostbuild compiles these device functions for the host: no PTX there)
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p + (unsigned)k * ls));
#else
    (void)k;
#endif
  }
};
// Layer loops are not unrolled: the step kernel is instruction-fetch sensitive (see step.cuh, SAMSIM_SYNC) and the
// loads of the next layers are already in flight through the L1 prefetches below.
#ifndef SAMSIM_LOOP
#define SAMSIM_LOOP _Pragma("unroll 1")
#endif
// Prefetch distance in layers, a per-handle run-time value (constant memory, samsim_b200_set_tuning); default 2.
#ifndef SAMSIM_PF
#define SAMSIM_PF (CFG.pf)
#endif

// elements between consecutive arrays of one layer of a tile (the 32 lanes); ARR_TILE*8 = 256 B
#define SAMSIM_TILE 32
// The per-layer views are built on the fly from two registers (base, ls) instead of being stored: 22 stored views
// were 350 B of local memory per thread and two local loads per access.  Functions copy the View out of the Col
// (`const View v = c`): Col lives in local memory (it is passed by reference through the call tree), and without the
// copy every layer iteration re-loaded base and ls from it.
struct View {
  double* base;    // &arr[tile][0][0][lane]
  unsigned ls;     // NA*32
  __device__ __forceinline__ Lay A(int id) const { return Lay{base + id * SAMSIM_TILE, ls}; }
  __device__ __forceinline__ Lay m() const { return A(AR_M); }
  __device__ __forceinline__ Lay S_abs() const { return A(AR_S_ABS); }
  __device__ __forceinline__ Lay H_abs() const { return A(AR_H_ABS); }
  __device__ __forceinline__ Lay thick() const { return A(AR_THICK); }
  __device__ __forceinline__ Lay T() const { return A(AR_T); }
  __device__ __forceinline__ Lay phi() const { return A(AR_PHI); }
  __device__ __forceinline__ Lay S_bu() const { return A(AR_S_BU); }
  __device__ __forceinline__ Lay psi_s() const { return A(AR_PSI_S); }
  __device__ __forceinline__ Lay psi_l() const { return A(AR_PSI_L); }
  __device__ __forceinline__ Lay psi_g() const { return A(AR_PSI_G); }
  __device__ __forceinline__ Lay ray() const { return A(AR_RAY); }
  __device__ __forceinline__ Lay perm() const { return A(AR_PERM); }
  __device__ __forceinline__ Lay flush_v() const { return A(AR_FLUSH_V); }
  __device__ __forceinline__ Lay flush_h() const { return A(AR_FLUSH_H); }
  __device__ __forceinline__ Lay fl_Q() const { return A(AR_FL_Q); }
  __device__ __forceinline__ Lay S_br() const { return A(AR_S_BR); }
  __device__ __forceinline__ Lay V_ex() const { return A(AR_V_EX); }
  __device__ __forceinline__ Lay fl_m() const { return A(AR_FL_M); }
  __device__ __forceinline__ Lay w0() const { return A(AR_W0); }
  __device__ __forceinline__ Lay w1() const { return A(AR_W1); }
  __device__ __forceinline__ Lay w2() const { return A(AR_W2); }
  __device__ __forceinline__ Lay w3() const { return A(AR_W3); }
  __device__ __forceinline__ Lay bgc(int q) const { return A(AR_BGC1 + q); }  // q = 0, 1
};
struct Col : View {
  double fb_x;  // fl_brine_bgc(N_active, 1): flooding (N_active >= 3; it is the up-cell of layer 1 when N_active == 2)
  int N_active, status, styropor_flag;
  unsigned ev0, ev1;  // branch events EV_* (bits 0..31 / 32..63), accumulated over the handle's lifetime
  // T, phi, S_bu of layers 2..N_active still equal what the S18 sweep of the previous step produced and
  // m, S_abs, H_abs of those layers are untouched since: the S4 sweep may reuse them (bit-identical result)
  bool thermo_valid;
  // last step of the launch: arrays that are only observable through get_array (fl_Q(2:)) are written
  bool want_state;
  // func_freeboard memo (see freeboard_of): everything here is a value the reference would recompute identically
  struct FbMemo {
    bool tot_valid;  double t1, A, G;          // forward totals SUM(psi_s*thick), SUM(psi_g*thick) for thick(1) == t1
    bool suf_valid;  int ks; double As, Gs;    // exact forward sums over layers ks+1..N_active
    bool res_valid;  double m1, th1, msnow, result;  // last result and the layer-1 / snow inputs it was computed from
    int k_last;                                // waterline layer of the last evaluation (start guess for the next step)
  } fb;
  // order-independent minima gathered by sweeps that read the data anyway (S24 health check, mo_grotz.f90:808-819)
  double min_psi_s, min_S_abs_2;
  // What the S18 sweep of the previous step prepared for the merged forward pass of this step (step.cuh,
  // backward_pass / forward_pass): gravity-drainage quantities of layers 2..N_active that depend only on T, phi, m,
  // thick, S_abs of those layers.  Valid while c.thermo_valid holds (nothing touched layers >= 2 since).
  struct Pre {
    bool valid;
    double mn2, sq2, st2;                 // layers 2..N_active-1: min(perm), ~SUM(thick/perm), ~SUM(thick) (suffix, backward order)
    double bottom_h, S_br_Na, perm_Na;    // thick(Na)*psi_s(Na)/psi_s_min, S_br(Na), perm(Na) as S4 / fl_grav_drain will see them
    double A2;                            // ~SUM(psi_s(2:Na)*thick(2:Na)): lower-bound certificate that the ice floats (S11)
  } pre;
  double sc[SC_COUNT];
  // clock (shared by the batch, advanced in lock step)
  double time;
  long long i;
  int n_time_out, time_counter;
  // forcing of this column for the current step (filled by the kernel's S1)
  double fsw0, fsw1, flw0, flw1;  // records time_counter-1 and time_counter, scaled
  double ftime0, ftime1;
};

#define SCV(c, id) ((c).sc[id])
#define EVT(c, id) (((id) < 32) ? ((c).ev0 |= (1u << ((id) & 31))) : ((c).ev1 |= (1u << ((id) & 31))))

__device__ __forceinline__ double f_max(double a, double b) { return (a > b) ? a : b; }  // Fortran MAX
__device__ __forceinline__ double f_min(double a, double b) { return (a < b) ? a : b; }  // Fortran MIN
__device__ __forceinline__ double f_sign(double a, double b) {                           // Fortran SIGN(a,b)
  return (dm_bits(b) < 0) ? -fabs(a) : fabs(a);
}
__device__ __forceinline__ double P2(double x) { return x * x; }
__device__ __forceinline__ double P3(double x) { return (x * x) * x; }
__device__ __forceinline__ double P4(double x) { double x2 = x * x; return x2 * x2; }

// ==========================================================================================
// mo_thermo_functions.f90
// ==========================================================================================

// func_S_br(T), mo_thermo_functions.f90:308-351 (c1 = 0 is added first, as in the source)
__device__ __forceinline__ double S_br_of(double T) {
  return 0.0 + CFG.c2 * T + CFG.c3 * P2(T) + CFG.c4 * P3(T);
}
// func_S_br(T,S_bu): clamp to >= S_bu, :353-357
__device__ __forceinline__ double S_br_of(double T, double S_bu) {
  double s = S_br_of(T);
  return (s < S_bu) ? S_bu : s;
}
// func_ddT_S_br, :380-414
__device__ __forceinline__ double ddT_S_br_of(double T) {
  const double T_crit = -20.0;
  double d = CFG.d2 + CFG.d3x2 * T + CFG.d4x3 * P2(T);
  if (T < T_crit) d = CFG.d2 + CFG.d3x2 * T_crit + CFG.d4x3 * P2(T_crit);
  return d;
}

// getT, mo_thermo_functions.f90:62-143: Newton for the freezing point, then Newton for T.
// `phi` keeps its incoming value when no branch assigns it (cannot happen for finite input).
//
// The reference computes the freezing point T_fr (:85-92) before every mushy inversion, but reads it only when an
// iterate leaves [-200, 0] degC (:101-103).  T_fr depends on S_bu alone and computing it has no side effect, so it
// is evaluated here on first use: same bits whenever the reference terminates, 11 of the ~25 divisions of a call gone.
// `ev1` receives the EV_GETT_* branch bits (word 1).
__device__ __forceinline__ double getT_freezing_point(double S_bu) {
  double T_fr = -1.0;
  while (fabs(S_br_of(T_fr) / S_bu - 1.0) > SAMSIM_F32(0.0001)) {  // :87
    const double T_0 = T_fr;
    const double f = S_br_of(T_0) - S_bu;
    const double ddT_f = ddT_S_br_of(T_0);
    T_fr = T_0 - f / ddT_f;
  }
  return T_fr;
}
// Returns false in the one case where the reference leaves phi untouched (salt-free branch with a NaN enthalpy):
// the caller then keeps the value the array holds.
__device__ __forceinline__ bool getT_body(double H, double S_bu, double T_in, double& T_out, double& phi,
                                          int& status, unsigned& ev1) {
  bool assigned = true;
  double T = H / c_l;
  if (S_br_of(T, S_bu) > S_bu && S_bu > 0.001) {
    double T_0, f, ddT_f;
    T_0 = T_in;
    {
      double sb = S_br_of(T_0);
      f = -latent_heat - H + latent_heat * S_bu / f_max(sb, 0.000000001) + c_s * T_0 + c_s_beta * T_0 * T_0 / 2.0;  // :95
      ddT_f = c_s + c_s_beta * T_0 - latent_heat * S_bu * ddT_S_br_of(T_0) / f_max(P2(sb), 0.0000000001);      // :96
    }
    T = T_0 - f / ddT_f;
    int it = 0;
    while (fabs(f) > 1.0) {  // :99
      T_0 = T;
      if (T_0 > 0.0 || T_0 < -200.0) {  // :101-103
        T_0 = getT_freezing_point(S_bu);
        ev1 |= 1u << (EV_GETT_TFR_FALLBACK - 32);
      }
      double sb = S_br_of(T_0);
      f = -latent_heat - H + latent_heat * S_bu / f_max(sb, 0.0000000001) + c_s * T_0 + c_s_beta * T_0 * T_0 / 2.0;  // :104
      ddT_f = c_s + c_s_beta * T_0 - latent_heat * S_bu * ddT_S_br_of(T_0) / f_max(sb * sb, 0.0000000001);       // :105
      T = T_0 - f / ddT_f;
      it++;
      if (it == 260) {  // :114-123 STOP 99
        status = 99;
        break;
      }
    }
    phi = 1.0 - S_bu / S_br_of(T, S_bu);  // :125
  } else if (S_bu < 0.001) {  // :127-137 salt-free
    ev1 |= 1u << (EV_GETT_SALTFREE - 32);
    if (H > 0.0) {
      phi = 0.0;
      T = H / c_l;
    } else if (H <= -latent_heat) {
      phi = 1.0;
      T = (H + latent_heat) / c_s;
    } else if (H <= 0.0 && -latent_heat < H) {
      T = 0.0;
      phi = -H / latent_heat;
    } else {
      assigned = false;
    }
  } else {
    ev1 |= 1u << (EV_GETT_LIQUID - 32);
    phi = 0.0;
  }
  T_out = T;
  return assigned;
}
// out-of-line copy for the call sites outside the two Newton sweeps (snow, coupling, layer 1)
__device__ __noinline__ void getT(double H, double S_bu, double T_in, double& T_out, double& phi,
                                  int& status, unsigned& ev1) {
  getT_body(H, S_bu, T_in, T_out, phi, status, ev1);
}

// Expulsion, mo_thermo_functions.f90:157-187
__device__ __forceinline__ void expulsion(double phi, double thick, double m, double& psi_s, double& psi_l,
                                          double& psi_g, double& V_ex) {
  double V_s = m * phi / rho_s;
  double V_l = m * (1.0 - phi) / rho_l;
  if (V_s + V_l > thick) V_ex = V_l + V_s - thick; else V_ex = 0.0;
  psi_s = V_s / thick;
  psi_l = (V_l - V_ex) / thick;
  psi_g = (thick - V_l - V_s + V_ex) / thick;
  if (psi_l < 0.0) psi_l = 0.0;
  if (psi_g < 0.0) psi_g = 0.0;
}

// sub_fl_Q, :201-224
__device__ __forceinline__ double fl_Q_between(double ps1, double pl1, double pg1, double th1, double T1, double ps2,
                                               double pl2, double pg2, double th2, double T2) {
  double k1 = ps1 * k_s + pl1 * k_l + pg1 * 0.0;
  double k2 = ps2 * k_s + pl2 * k_l + pg2 * 0.0;
  double R = th1 / (2.0 * k1) + th2 / (2.0 * k2);
  return (T2 - T1) / R;
}
// sub_fl_Q_0 with direct_flag = -1 (the only value any call site passes), :238-265
__device__ __forceinline__ double fl_Q_0_top(double ps, double pl, double pg, double th, double T, double T_bound) {
  double k = ps * k_s + pl * k_l + pg * 0.0;
  double R = th / (2.0 * k);
  return (T - T_bound) / R;
}

// ==========================================================================================
// mo_functions.f90
// ==========================================================================================

// func_density, mo_functions.f90:51-62
__device__ __forceinline__ double density_of(double T, double S) {
  double density_0 = 999.842594 + 6.8 / 100.0 * T;
  return density_0 + 0.825 * S + (-5.7 / 1000.0) * det_pow(f_max(S, 0.0), 1.5);
}

// func_T_freeze, :239-250
__device__ __forceinline__ double T_freeze_of(double S_bu, int salt_flag) {
  double Tf = 0.0;
  if (salt_flag == 2) {
    const double c2 = (double)9.37f;
    const double c3 = (double)(5.33f * 1e-7f);
    Tf = -0.0592 * S_bu - c2 * P2(S_bu) - c3 * P3(S_bu);
  } else if (salt_flag == 1) {
    const double a = (double)(1.710523f * 1e-3f);
    const double b = (double)(2.154996f * 1e-4f);
    Tf = -0.0575 * S_bu + a * det_pow(S_bu, 1.5) - b * P2(S_bu);
  }
  return Tf;
}

// func_albedo, :157-208
__device__ __forceinline__ double albedo_of(double thick_snow, double T_snow, double psi_l, double thick_min,
                                            int albedo_flag) {
  const double ice_dry = SAMSIM_F32(0.75), ice_wet = SAMSIM_F32(0.6), snow_dry = SAMSIM_F32(0.85),
               snow_wet = SAMSIM_F32(0.75), water = SAMSIM_F32(0.2);
  double albedo;
  if (thick_snow > thick_min) {
    albedo = (T_snow < SAMSIM_F32(-0.01)) ? snow_dry : snow_wet;
    albedo = ice_dry + (albedo - ice_dry) * f_min(1.0, thick_snow / 0.3);
  } else {
    if (psi_l > 0.9) albedo = water;
    else if (psi_l > 0.6) albedo = ice_wet + (water - ice_wet) * ((psi_l - 0.6) / 0.3);
    else if (psi_l > 0.2) albedo = ice_wet;
    else albedo = ice_dry;
  }
  if (albedo_flag == 1) {
    if (thick_snow > thick_min) albedo = (T_snow < SAMSIM_F32(-0.01)) ? snow_dry : snow_wet;
    else albedo = (psi_l < SAMSIM_F32(0.8)) ? ice_dry : water;
  }
  return albedo;
}

// func_k_snow, mo_snow.f90:560-573
__device__ __forceinline__ double k_snow_of(double m_snow, double thick_snow) {
  const double c0 = 0.138, c1 = -1.01 / 1000.0, c2 = 3.233 / 1000000.0;
  double r = m_snow / thick_snow;
  double k = c0 + c1 * m_snow / thick_snow + c2 * P2(r);
  return k + SAMSIM_F32(0.15);
}

// sub_notzflux, mo_functions.f90:270-289
__device__ __forceinline__ void notzflux(double time, double& fl_sw, double& fl_rest) {
  double day = time / 86400.0;
  while (day > 360) day = day - 360;
  fl_sw = 314.0 * det_exp(-0.5 * P2((day - 164.0) / SAMSIM_F32(47.9)));
  fl_rest = 118.0 * det_exp(-0.5 * P2((day - 206.0) / SAMSIM_F32(53.1))) + 179.0;
  if (day < 60. || day > 300.) fl_sw = 0.0;
}

// forward sums in the reference's order: SUM(a(i:j)) and SUM(a(i:j)*b(i:j))
// Four layers are loaded before they are added (one after the other, in order): four loads in flight per thread
// instead of one; the sums are latency-bound otherwise.
#ifdef SAMSIM_SUM_NOINLINE
#define SAMSIM_SUM_ATTR __noinline__
#else
#define SAMSIM_SUM_ATTR __forceinline__
#endif
__device__ SAMSIM_SUM_ATTR double sum_fwd(const Lay& a, int i, int j) {
  double s = 0.0;
  int q = i;
  SAMSIM_LOOP
  for (; q + 3 <= j; q += 4) {
    const double a0 = a[q], a1 = a[q + 1], a2 = a[q + 2], a3 = a[q + 3];
    s = s + a0; s = s + a1; s = s + a2; s = s + a3;
  }
  SAMSIM_LOOP
  for (; q <= j; q++) s = s + a[q];
  return s;
}
__device__ SAMSIM_SUM_ATTR double sum_prod_fwd(const Lay& a, const Lay& b, int i, int j) {
  double s = 0.0;
  int q = i;
  SAMSIM_LOOP
  for (; q + 3 <= j; q += 4) {
    const double a0 = a[q], a1 = a[q + 1], a2 = a[q + 2], a3 = a[q + 3];
    const double b0 = b[q], b1 = b[q + 1], b2 = b[q + 2], b3 = b[q + 3];
    s = s + a0 * b0; s = s + a1 * b1; s = s + a2 * b2; s = s + a3 * b3;
  }
  SAMSIM_LOOP
  for (; q <= j; q++) s = s + a[q] * b[q];
  return s;
}

// func_freeboard, mo_functions.f90:79-130.
// The reference recomputes test2(k) = SUM(psi_s(k+1:Na)*thick(k+1:Na))*(rho_l-rho_s) + SUM(psi_g(..)*thick(..))*rho_l
// with fresh forward sums for every k of its DO WHILE (O(N k)).  Only the value at the k where the loop stops is
// used; for the earlier k only the outcome of `test1 < test2` matters.  Here the outcome is decided from
// total - prefix (equal to the forward sum up to a rounding error bounded far below `margin`); the exact forward
// sum is evaluated only where the decision is within the margin or the loop stops, so the returned value is the
// reference's, bit for bit, at O(N) cost.
// Memo: (1) the result is reused while its inputs are unchanged -- psi_s, psi_g, thick(2:), m(2:) only change at
// S4/S5 and at flood/flush/layer events (which reset the memo), so between the calls of one step only m(1),
// thick(1), m_snow can differ and they are compared; (2) the forward totals are reused while thick(1) is unchanged;
// (3) the exact suffix sums for waterline layer ks are reused.  (2) and (3) are pre-filled by the fused S4 pass.
__device__ __noinline__ double freeboard_of(Col& c) {
  const View v = c;
  const int Na = c.N_active;
  const double snowmass = (CFG.freeboard_snow_flag == 0) ? SCV(c, SC_M_SNOW) : 0.0;
  const double m1 = v.m()[1], th1 = v.thick()[1];
  Col::FbMemo& fb = c.fb;
  if (fb.res_valid && fb.m1 == m1 && fb.th1 == th1 && fb.msnow == snowmass) return fb.result;
  double A = 0.0, G = 0.0;
  bool have_totals = false;
  if (fb.tot_valid && fb.t1 == th1) {
    A = fb.A; G = fb.G;
    have_totals = true;
  } else if (fb.tot_valid) {
    // Only thick(1) moved since the totals were taken (S20 melts the surface every step of the melt season).  Swap
    // the first term: equal to the fresh forward sum up to a few ulps, far inside `margin`.  The totals are used
    // exactly only when the snow outweighs the buoyancy (:99-102), so this needs snowmass < buoy beyond the margin.
    const double ps1 = v.psi_s()[1], pg1 = v.psi_g()[1];
    const double A1 = fb.A - ps1 * fb.t1 + ps1 * th1, G1 = fb.G - pg1 * fb.t1 + pg1 * th1;
    const double b1 = A1 * (rho_l - rho_s) + G1 * rho_l;
    if (snowmass < b1 - (1e-9 * (fabs(b1) + fabs(snowmass)) + 1e-300)) { A = A1; G = G1; have_totals = true; }
  }
  if (!have_totals) {
    A = 0.0; G = 0.0;  // forward totals, the reference's order
    SAMSIM_LOOP
    for (int q = 1; q <= Na; q++) {
      if (q + SAMSIM_PF <= Na) { v.psi_s().prefetch(q + SAMSIM_PF); v.psi_g().prefetch(q + SAMSIM_PF); v.thick().prefetch(q + SAMSIM_PF); }
      const double t = v.thick()[q];
      A = A + v.psi_s()[q] * t;
      G = G + v.psi_g()[q] * t;
    }
    fb.tot_valid = true; fb.t1 = th1; fb.A = A; fb.G = G;
  }
  const double buoy = A * (rho_l - rho_s) + G * rho_l;
  double freeboard;
  if (snowmass > buoy) {  // :99-102 snow pushes the ice under water
    freeboard = buoy - snowmass;
    freeboard = freeboard / rho_l;
  } else {
    const double margin = 1e-9 * (fabs(buoy) + fabs(snowmass)) + 1e-300;
    double pA = 0.0, pG = 0.0, msum = 0.0, msum_prev = 0.0, test1 = 0.0, test2 = 1.0, thsum = 0.0, thsum_prev = 0.0;
    int k = 0;
    while (test1 < test2) {  // :114-118
      k = k + 1;
      const double t = v.thick()[k];
      pA = pA + v.psi_s()[k] * t;   // same partial sums as the forward totals above
      pG = pG + v.psi_g()[k] * t;
      msum_prev = msum;
      msum = msum + v.m()[k];       // SUM(m(1:k)): fixed-start prefix, incremental is the same order
      thsum_prev = thsum;
      thsum = thsum + t;            // SUM(thick(1:k)) likewise
      test1 = msum + snowmass;
      const double approx = (A - pA) * (rho_l - rho_s) + (G - pG) * rho_l;
      if (test1 < approx - margin) {
        test2 = approx + margin;    // certainly test1 < exact test2: keep looping (value unused)
      } else {
        if (!(fb.suf_valid && fb.ks == k)) {
          fb.As = sum_prod_fwd(v.psi_s(), v.thick(), k + 1, Na);
          fb.Gs = sum_prod_fwd(v.psi_g(), v.thick(), k + 1, Na);
          fb.ks = k; fb.suf_valid = true;
        }
        test2 = fb.As * (rho_l - rho_s) + fb.Gs * rho_l;
      }
    }
    fb.k_last = k;
    test1 = msum_prev + snowmass;  // :121 SUM(m(1:k-1))
    const double mk = v.m()[k], tk = v.thick()[k];
    freeboard = test2 - test1 + (rho_l - mk / tk) * tk;  // :124
    freeboard = freeboard / rho_l;
    freeboard = freeboard + thsum_prev;                  // :126 SUM(thick(1:k-1))
  }
  fb.res_valid = true; fb.m1 = m1; fb.th1 = th1; fb.msnow = snowmass; fb.result = freeboard;
  return freeboard;
}
// every change of psi_s / psi_g / thick(2:) / m(2:) / N_active goes through one of these
__device__ __forceinline__ void fb_reset(Col& c) { c.fb.tot_valid = false; c.fb.suf_valid = false; c.fb.res_valid = false; }

// sub_melt_thick, mo_functions.f90:386-428
// returns true when the gas-fraction correction (:418-426) ran (event bit only)
__device__ __forceinline__ bool melt_thick_of(double psi_l, double psi_s, double psi_g, double T, double T_freeze,
                                              double T_top, double fl_Q, double thick_snow, double dt,
                                              double& melt_thick, double& thick, double thick_min) {
  bool gas = false;
  melt_thick = 0.0;
  if (thick_snow < thick_min && T_top >= T_freeze) {
    melt_thick = -fl_Q - 2.0 * (psi_l * k_l + psi_s * k_s) / thick * (T_freeze - T);
    melt_thick = melt_thick * dt / f_max((latent_heat * rho_s * psi_s), 0.000000000000001);
    melt_thick = f_min(psi_l * thick, melt_thick);
  }
  if (psi_s < psi_s_top_min) melt_thick = thick * (1.0 - psi_s / psi_s_top_min);
  if (melt_thick > 0.0 && psi_g > gas_snow_ice2) {
    gas = true;
    if (melt_thick > (psi_g - gas_snow_ice2) * thick) {
      melt_thick = melt_thick - (psi_g - gas_snow_ice2) * thick;
      thick = thick * (1.0 - (psi_g - gas_snow_ice2));
    } else {
      thick = thick - melt_thick;
      melt_thick = 0.0;
    }
  }
  return gas;
}

// sub_melt_snow, mo_functions.f90:443-474; returns true when all the snow went into the ice (:453)
__device__ __forceinline__ bool melt_snow(double& melt_thick, double& thick, double& thick_snow, double& H_abs,
                                          double& H_abs_snow, double& m, double& m_snow, double& psi_g_snow) {
  double shift = 1.0 / f_max(psi_g_snow, 0.01) * melt_thick;
  if (shift >= thick_snow) {
    melt_thick = melt_thick - thick_snow * psi_g_snow;
    H_abs = H_abs + H_abs_snow;
    m = m + m_snow;
    thick = thick + (1.0 - psi_g_snow) * thick_snow;
    thick_snow = 0.0;
    m_snow = 0.0;
    H_abs_snow = 0.0;
    return true;
  } else {
    H_abs = H_abs + shift / thick_snow * H_abs_snow;
    H_abs_snow = H_abs_snow - shift / thick_snow * H_abs_snow;
    m = m + shift / thick_snow * m_snow;
    m_snow = m_snow - shift / thick_snow * m_snow;
    thick = thick + shift - melt_thick;
    thick_snow = thick_snow - shift;
    melt_thick = 0.0;
  }
  return false;
}

// ==========================================================================================
// mo_mass.f90
// ==========================================================================================

// One layer of mass_transfer, mo_mass.f90:76-95.  f1 = fl_m(k+1), f0 = fl_m(k); *_km1 / *_kp1 are the neighbours
// (TT, SS_bu, SS_abs of the reference; Sabs_km1 is the ALREADY UPDATED S_abs(k-1), :91).  H, S = H_abs(k), S_abs(k).
__device__ __forceinline__ void mass_transfer_layer(double f1, double f0, double T_km1, double Sbu_km1,
                                                    double Sabs_km1, double T_k, double Sbu_k, double T_kp1,
                                                    double Sbu_kp1, double Sabs_kp1, double& H, double& S) {
  if (f1 > 0.) {
    H = H + f1 * T_kp1 * c_l;
    S = S + f_min(f1 * S_br_of(T_kp1, Sbu_kp1), Sabs_kp1);
  } else if (f1 < 0.) {
    H = H + f1 * T_k * c_l;
    S = S + f_max(f1 * S_br_of(T_k, Sbu_k), -S);
  }
  if (f0 > 0.) {
    H = H - f0 * T_k * c_l;
    S = S - f_min(f0 * S_br_of(T_k, Sbu_k), S);
  } else if (f0 < 0) {
    H = H - f0 * T_km1 * c_l;
    S = S - f_max(f0 * S_br_of(T_km1, Sbu_km1), -Sabs_km1);
  }
}

// mass_transfer, mo_mass.f90:53-96, as ONE in-place forward pass.  The reference copies T, S_bu and
// S_abs into TT/SS_bu/SS_abs first; T and S_bu are not modified by the routine and SS_abs(k+1)
// is read before layer k+1 is updated, so reading the live arrays is equivalent.  S_abs(k-1)
// in the last branch IS the updated value in the reference too (:91).
// `kstart`: the caller guarantees fl_m(1:kstart) == 0, so layers 1..kstart-1 are left untouched (both of their
// faces carry no flux) and the pass starts at kstart; with kstart > 1 the carried neighbour values are loaded.
__device__ __noinline__ void mass_transfer(Col& c, const Lay& fl_m, const Lay& S_bu_view, int kstart = 1) {
  const View v = c;
  const int Na = c.N_active;
  const double T_bottom = SCV(c, SC_T_BOTTOM), S_bu_bottom = SCV(c, SC_S_BU_BOTTOM);
  if (kstart < 1) kstart = 1;
  if (kstart > Na) return;
  double T_km1 = 0.0, Sbu_km1 = 0.0, Sabs_km1 = 0.0;  // k = 1: fl_m(1) == 0 at every call site, never read
  if (kstart > 1) { T_km1 = v.T()[kstart - 1]; Sbu_km1 = S_bu_view[kstart - 1]; Sabs_km1 = v.S_abs()[kstart - 1]; }
  double T_k = v.T()[kstart], Sbu_k = S_bu_view[kstart];
  double f0 = fl_m[kstart];
  SAMSIM_LOOP
  for (int k = kstart; k <= Na; k++) {
    if (k + SAMSIM_PF <= Na) {
      v.T().prefetch(k + SAMSIM_PF); S_bu_view.prefetch(k + SAMSIM_PF); v.S_abs().prefetch(k + SAMSIM_PF);
      v.H_abs().prefetch(k + SAMSIM_PF); fl_m.prefetch(k + SAMSIM_PF);
    }
    double T_kp1, Sbu_kp1, Sabs_kp1;
    if (k < Na) {
      T_kp1 = v.T()[k + 1];
      Sbu_kp1 = S_bu_view[k + 1];
      Sabs_kp1 = v.S_abs()[k + 1];
    } else {
      T_kp1 = T_bottom;
      Sbu_kp1 = S_bu_bottom;
      Sabs_kp1 = S_bu_bottom * 2000.0;
    }
    const double f1 = fl_m[k + 1];
    double H = v.H_abs()[k], S = v.S_abs()[k];
    mass_transfer_layer(f1, f0, T_km1, Sbu_km1, Sabs_km1, T_k, Sbu_k, T_kp1, Sbu_kp1, Sabs_kp1, H, S);
    v.H_abs()[k] = H;
    v.S_abs()[k] = S;
    T_km1 = T_k; Sbu_km1 = Sbu_k; Sabs_km1 = S;
    T_k = T_kp1; Sbu_k = Sbu_kp1;
    f0 = f1;
  }
}

// ==========================================================================================
// mo_snow.f90
// ==========================================================================================

// snow_coupling, mo_snow.f90:61-104.  The reference's getT calls alias T_in with T, which makes
// the first guess H/c_l (SURVEY section 7); passed explicitly here.
__device__ __noinline__ void snow_coupling(Col& c, double& H_abs1, double& phi1, double& T1, double m1,
                                           double S_bu1) {
  const View v = c;
  double& H_abs_snow = SCV(c, SC_H_ABS_SNOW);
  double& phi_s = SCV(c, SC_PHI_S);
  double& T_snow = SCV(c, SC_T_SNOW);
  const double m_snow = SCV(c, SC_M_SNOW), S_abs_snow = SCV(c, SC_S_ABS_SNOW);
  H_abs1 = H_abs1 + m_snow * latent_heat + H_abs_snow;
  H_abs_snow = -m_snow * latent_heat;
  double H = H_abs1 / m1;
  double hs = H_abs_snow / m_snow;
  getT(hs, S_abs_snow / m_snow, hs / c_l, T_snow, phi_s, c.status, c.ev1);
  getT(H, S_bu1, H / c_l, T1, phi1, c.status, c.ev1);
  if (T1 > 0 && H_abs1 <= -H_abs_snow) {
    EVT(c, EV_SNOW_COUPLING_WARM1);
    H_abs_snow = H_abs_snow + H_abs1;
    H_abs1 = 0.0;
    hs = H_abs_snow / m_snow;
    getT(hs, S_abs_snow / m_snow, hs / c_l, T_snow, phi_s, c.status, c.ev1);
    getT(H, S_bu1, H / c_l, T1, phi1, c.status, c.ev1);  // H is NOT refreshed here in the reference (:79-80)
  } else if (T1 > 0. && H_abs1 > -H_abs_snow) {
    EVT(c, EV_SNOW_COUPLING_WARM2);
    H_abs1 = (H_abs1 + H_abs_snow) * m1 / m_snow / (1.0 + m1 / m_snow);
    H_abs_snow = H_abs1 * m_snow / m1;
    hs = H_abs_snow / m_snow;
    getT(hs, S_abs_snow / m_snow, hs / c_l, T_snow, phi_s, c.status, c.ev1);
    getT(H, S_bu1, H / c_l, T1, phi1, c.status, c.ev1);
  } else {
    int jj = 0;
    while (fabs(T1 - T_snow) > SAMSIM_F32(0.1) && jj < 201) {
      double d = T_snow - (T_snow + T1) / 2.0;
      double step = f_sign(f_max(fabs(d), 0.1), d) * c_s * m_snow;
      H_abs_snow = H_abs_snow - step;
      H_abs1 = H_abs1 + step;
      jj = jj + 1;
      EVT(c, EV_SNOW_COUPLING_ITER);
      H = H_abs1 / m1;
      hs = H_abs_snow / m_snow;
      getT(hs, S_abs_snow / m_snow, hs / c_l, T_snow, phi_s, c.status, c.ev1);
      getT(H, S_bu1, H / c_l, T1, phi1, c.status, c.ev1);
      if (c.status) return;
    }
    if (jj > 200 && fabs(T1 - T_snow) > 1.0) c.status = 16;
  }
}

// snow_precip, mo_snow.f90:123-150 (have_solid: precip_flag 0 passes solid_precip)
__device__ __forceinline__ void snow_precip(Col& c, double dt, double liquid_in, double T2m, bool have_solid,
                                            double solid_in) {
  const View v = c;
  double solid, liquid;
  if (have_solid) { solid = solid_in; liquid = liquid_in; }
  else if (T2m > 0.0) { solid = 0.0; liquid = liquid_in; }
  else { solid = liquid_in; liquid = 0.0; }
  double d_thick = dt * solid * rho_l / rho_snow;
  SCV(c, SC_M_SNOW) = SCV(c, SC_M_SNOW) + dt * rho_l * (liquid + solid);
  SCV(c, SC_THICK_SNOW) = SCV(c, SC_THICK_SNOW) + d_thick;
  double H = SCV(c, SC_H_ABS_SNOW);
  H = H + dt * T2m * liquid * rho_l * c_l;
  H = H + dt * f_min(T2m, -1.0) * solid * rho_l * c_s;
  H = H - dt * solid * rho_l * latent_heat;
  SCV(c, SC_H_ABS_SNOW) = H;
}

// snow_precip_0, mo_snow.f90:167-192
__device__ __forceinline__ void snow_precip_0(double& H_abs, double& S_abs, double m, double T, double dt,
                                              double liquid_in, double T2m, bool have_solid, double solid_in) {
  double solid, liquid;
  if (have_solid) { solid = solid_in; liquid = liquid_in; }
  else if (T2m > 0.0) { solid = 0.0; liquid = liquid_in; }
  else { solid = liquid_in; liquid = 0.0; }
  H_abs = H_abs + (liquid + solid) * (T2m - T) * dt;
  H_abs = H_abs - solid * latent_heat * dt;
  S_abs = S_abs - (liquid + solid) * S_abs / m * dt;
}

// snow_thermo (mo_snow.f90:212-319) and snow_thermo_meltwater (:331-458) share everything up to
// the saturated-layer block; `meltwater` selects the variant.
__device__ __noinline__ void snow_thermo(Col& c, bool meltwater, double& m1, double& thick1,
                                         double& H_abs1, double& melt_thick_snow) {
  const View v = c;
  double& psi_l_snow = SCV(c, SC_PSI_L_SNOW);
  double& psi_s_snow = SCV(c, SC_PSI_S_SNOW);
  double& psi_g_snow = SCV(c, SC_PSI_G_SNOW);
  double& thick_snow = SCV(c, SC_THICK_SNOW);
  double& S_abs_snow = SCV(c, SC_S_ABS_SNOW);
  double& H_abs_snow = SCV(c, SC_H_ABS_SNOW);
  double& m_snow = SCV(c, SC_M_SNOW);
  double& T_snow = SCV(c, SC_T_SNOW);
  double phi_snow = 0.0, max_lwc, max_lwc_v, sat_snow;

  const double H_snow = H_abs_snow / m_snow;
  const double S_bu_snow = S_abs_snow / m_snow;
  const double psi_s_old = psi_s_snow;
  if (meltwater) EVT(c, EV_SNOW_THERMO_MELTWATER); else EVT(c, EV_SNOW_THERMO);
  {
    double T_in = T_snow;
    getT(H_snow, S_bu_snow, T_in, T_snow, phi_snow, c.status, c.ev1);
  }
  psi_s_snow = m_snow * phi_snow / rho_s / thick_snow;
  psi_l_snow = m_snow * (1.0 - phi_snow) / rho_l / thick_snow;
  if (psi_s_snow + psi_l_snow > 1.0) {
    thick_snow = m_snow * (phi_snow / rho_s + (1.0 - phi_snow) / rho_l);
    psi_s_snow = m_snow * phi_snow / rho_s / thick_snow;
    psi_l_snow = m_snow * (1.0 - phi_snow) / rho_l / thick_snow;
    if (fabs(psi_s_snow + psi_l_snow - 1.0) > 0.0000001) { c.status = 345; return; }
  }
  psi_g_snow = 1.0 - psi_s_snow - psi_l_snow;
  if (psi_s_snow > 0.0) max_lwc = 0.057 * (1.0 - psi_s_snow) / (psi_s_snow) + 0.017;
  else max_lwc = 0.0;

  if (psi_s_old > psi_s_snow && psi_s_snow > 0.0) {
    EVT(c, EV_SNOW_COMPACTION);
    if ((1.0 - phi_snow) > max_lwc) thick_snow = thick_snow * (1.0 - (psi_s_old - psi_s_snow) / psi_s_old);
    if (thick_snow < (phi_snow * m_snow / rho_s + (1.0 - phi_snow) * m_snow / rho_l))
      thick_snow = (phi_snow * m_snow / rho_s + (1.0 - phi_snow) * m_snow / rho_l);
    psi_s_snow = m_snow * phi_snow / rho_s / thick_snow;
    psi_l_snow = m_snow * (1.0 - phi_snow) / rho_l / thick_snow;
    psi_g_snow = 1.0 - psi_s_snow - psi_l_snow;
    psi_g_snow = fabs(psi_g_snow);
  } else if (psi_s_snow < 0.000001) {
    thick_snow = m_snow / rho_l;
    psi_s_snow = 0.0;
    psi_g_snow = 0.0;
    psi_l_snow = 1.0;
  }

  const bool wet = meltwater ? ((1.0 - phi_snow) > max_lwc && psi_l_snow > 0.0 && psi_g_snow > 0.0)
                             : ((1.0 - phi_snow) > max_lwc && psi_g_snow > 0.0);
  if (wet) {
    EVT(c, EV_SNOW_WET);
    max_lwc_v = max_lwc * m_snow / (rho_l * thick_snow);
    if (!meltwater) {  // mo_snow.f90:272-294
      sat_snow = thick_snow * (psi_l_snow - max_lwc_v);
      sat_snow = sat_snow / (1.0 - psi_s_snow - max_lwc_v - f_min(gas_snow_ice2, psi_g_snow));
      thick_snow = thick_snow - sat_snow;
      thick1 = thick1 + sat_snow;
      m_snow = m_snow - sat_snow * (psi_s_snow * rho_s + (1.0 - psi_s_snow - gas_snow_ice2) * rho_l);
      m1 = m1 + sat_snow * (psi_s_snow * rho_s + (1.0 - psi_s_snow - gas_snow_ice2) * rho_l);
      H_abs_snow = H_abs_snow - sat_snow * psi_s_snow * rho_s * c_s * T_snow;
      H_abs1 = H_abs1 + sat_snow * psi_s_snow * rho_s * c_s * T_snow;
      H_abs_snow = H_abs_snow + sat_snow * psi_s_snow * rho_s * latent_heat;
      H_abs1 = H_abs1 - sat_snow * psi_s_snow * rho_s * latent_heat;
      H_abs_snow = H_abs_snow - sat_snow * (1.0 - psi_s_snow) * rho_l * c_l * T_snow;
      H_abs1 = H_abs1 + sat_snow * (1.0 - psi_s_snow) * rho_l * c_l * T_snow;
    } else {  // :399-430
      const double slush = (psi_l_snow - max_lwc_v) * (1.0 - CFG.k_snow_flush);
      const double flush = (psi_l_snow - max_lwc_v) * CFG.k_snow_flush;
      melt_thick_snow = thick_snow * flush;
      sat_snow = thick_snow * (slush);
      sat_snow = sat_snow / (1.0 - psi_s_snow - max_lwc_v - f_min(gas_snow_ice2, psi_g_snow));
      const double gg = f_min(gas_snow_ice2, psi_g_snow);
      thick_snow = thick_snow - sat_snow - melt_thick_snow;
      thick1 = thick1 + sat_snow;
      m_snow = m_snow - sat_snow * (psi_s_snow * rho_s + (1.0 - psi_s_snow - gg) * rho_l) - melt_thick_snow * rho_l;
      m1 = m1 + sat_snow * (psi_s_snow * rho_s + (1.0 - psi_s_snow - gg) * rho_l);
      H_abs_snow = H_abs_snow - sat_snow * psi_s_snow * rho_s * c_s * T_snow;
      H_abs1 = H_abs1 + sat_snow * psi_s_snow * rho_s * c_s * T_snow;
      H_abs_snow = H_abs_snow + sat_snow * psi_s_snow * rho_s * latent_heat;
      H_abs1 = H_abs1 - sat_snow * psi_s_snow * rho_s * latent_heat;
      H_abs_snow = H_abs_snow - sat_snow * (1.0 - psi_s_snow - gg) * rho_l * c_l * T_snow -
                   melt_thick_snow * rho_l * c_l * T_snow;
      H_abs1 = H_abs1 + sat_snow * (1.0 - psi_s_snow - gg) * rho_l * c_l * T_snow;
    }
  } else if (psi_g_snow <= 0.0) {
    EVT(c, EV_SNOW_MERGE);
    H_abs1 = H_abs1 + H_abs_snow;
    m1 = m1 + m_snow;
    thick1 = thick1 + thick_snow;
    H_abs_snow = 0.0; m_snow = 0.0; thick_snow = 0.0;
    psi_g_snow = 0.0; psi_s_snow = 0.0; psi_l_snow = 0.0;
  }
  if (psi_g_snow < 0.0) c.status = 9876;
}

// the driver's snow block, mo_grotz.f90:273-292 and :601-621
__device__ __forceinline__ void snow_block(Col& c) {
  const View v = c;
  if (SCV(c, SC_THICK_SNOW) > 0.0) {
    double m1 = v.m()[1], th1 = v.thick()[1], H1 = v.H_abs()[1];
    if (CFG.snow_flush_flag == 0) {
      double dummy = 0.0;
      snow_thermo(c, false, m1, th1, H1, dummy);
      SCV(c, SC_MELT_THICK_SNOW) = 0.0;
    } else if (CFG.snow_flush_flag == 1) {
      SCV(c, SC_MELT_THICK_SNOW) = 0.0;
      snow_thermo(c, true, m1, th1, H1, SCV(c, SC_MELT_THICK_SNOW));
    }
    v.m()[1] = m1; v.thick()[1] = th1; v.H_abs()[1] = H1;
  } else {
    SCV(c, SC_THICK_SNOW) = 0.0; SCV(c, SC_M_SNOW) = 0.0; SCV(c, SC_PSI_S_SNOW) = 0.0; SCV(c, SC_PSI_L_SNOW) = 0.0;
    SCV(c, SC_PSI_G_SNOW) = 0.0; SCV(c, SC_H_ABS_SNOW) = 0.0; SCV(c, SC_S_ABS_SNOW) = 0.0;
    SCV(c, SC_MELT_THICK_SNOW) = 0.0;
  }
}

// sub_fl_Q_0_snow_thin :466-487, sub_fl_Q_snow :498-518, sub_fl_Q_0_snow :528-545
__device__ __forceinline__ double fl_Q_0_snow_thin(double m_snow, double thick_snow, double T_snow, double ps,
                                                   double pl, double pg, double thick, double T_bound) {
  double ks = k_snow_of(m_snow, thick_snow);
  double k = ps * k_s + pl * k_l + pg * 0.0;
  k = thick_snow / (thick_snow + thick) * ks + thick / (thick_snow + thick) * k;
  double R = (thick_snow + thick) / (2.0 * k);
  return (T_snow - T_bound) / R;
}
__device__ __forceinline__ double fl_Q_snow_ice(double m_snow, double thick_snow, double T_snow, double ps2,
                                                double pl2, double th2, double T2) {
  double ks = k_snow_of(m_snow, thick_snow);
  double k2 = ps2 * k_s + pl2 * k_l;
  double R = thick_snow / (2.0 * ks) + th2 / (2.0 * k2);
  return (T2 - T_snow) / R;
}
__device__ __forceinline__ double fl_Q_0_snow(double m_snow, double thick_snow, double T_snow, double T_bound) {
  double k = k_snow_of(m_snow, thick_snow);
  double R = thick_snow / (2.0 * k);
  return (T_snow - T_bound) / R;
}

// ==========================================================================================
// mo_grav_drain.f90
// ==========================================================================================

// fl_grav_drain, mo_grav_drain.f90:74-201.  Scratch: w0 perm, w1 thick/perm, w2 suffix-min(perm), fl_m.
//
// The reference evaluates, for every layer k, SUM_{kk=k}^{Na-1} thick(kk)/perm(kk) and SUM(thick(k:Na-1)) as fresh
// forward sums (O(N^2), :115-120) and SUM(thick(k+1:Na-1)) for the height (:128).  Forward order is part of the
// arithmetic contract, so the sums are kept as they are but evaluated for GB consecutive k at once with the GB
// accumulators in registers: every thick/perm value is loaded once per block instead of once per k.
// SUM(thick(k+1:Na-1)) of layer k is the same forward sum as SUM(thick(k':Na-1)) of layer k' = k+1.
// The FORALL fl_up(k:N_active) += flux (:162-164) is a running sum in layer order; only element k is clamped
// (:166), which the carry does not see -- same additions, O(N).
//
// Lazy Rayleigh numbers (exact_all == false).  ray(k) is observable only through the S8 record of the NEXT step
// and through get_array after the launch; on every other step it matters only where it can exceed ray_crit (:145).
// The backward pass therefore also accumulates the two sums as plain suffix sums (same terms, other order:
// relative deviation <= ~1e-14) and classifies every layer with them; the reference's forward sums are evaluated
// only for layers whose estimate is above ray_crit*(1 - 1e-10) -- a margin four orders wider than the deviation --
// so decisions and fluxes are the reference's, bit for bit, and layers that cannot drain cost O(1).
// With harmonic_flag 2 and no tracers, a cheaper bound pass first rules out the layers above the topmost layer
// whose estimate can come near ray_crit (in mid-winter the warm bottom fifth): they need no det_pow and no
// division, and keep ray from an earlier step, which nothing reads before an exact_all step rewrites it.
#ifndef SAMSIM_GB
#define SAMSIM_GB 8   // layers per block of the blocked forward sums: 16 accumulators in registers
#endif
// Bound pass of grav_drain (harmonic_flag 2): the estimate with thick/perm from below (dm_perm_inv_lo) and no
// division, est > thr tested as P*(st + bottom_h) > thr*(kappa_l*mu)*(sq + qb).  Every layer whose estimate exceeds
// ray_crit*(1 - 1e-10) is flagged, and so is any comparison with a NaN (DESIGN §5.1).  Nothing is stored.  Returns
// the first layer of the block of the blocked sums (SAMSIM_GB) that holds the topmost flagged layer, or Na when no
// layer is flagged.  Out of line: its registers stay out of grav_drain's allocation.
__device__ __noinline__ int grav_drain_bound(const Col& c, double bottom_h, double S_br_Na) {
  const View v = c;
  const int Na = c.N_active;
  const double thr = (ray_crit * (1.0 - 1e-6)) * (kappa_l * mu);
  double sq = 0.0, st = 0.0, qb = 0.0;
  int ktop = 0;  // topmost flagged layer
  SAMSIM_LOOP
  for (int k = Na; k >= 1; k--) {
    if (k - SAMSIM_PF >= 1) { v.psi_l().prefetch(k - SAMSIM_PF); v.thick().prefetch(k - SAMSIM_PF); v.S_br().prefetch(k - SAMSIM_PF); }
    const double ip = dm_perm_inv_lo(v.psi_l()[k]);
    if (k == Na) { qb = bottom_h * ip; continue; }
    const double thk = v.thick()[k];
    const double st_below = st;
    sq = sq + thk * ip;
    st = st + thk;
    const double a = grav * rho_l * bbeta * (v.S_br()[k] - S_br_Na) * (st_below + bottom_h) * (st + bottom_h);
    if (!(a <= thr * (sq + qb))) ktop = k;
  }
  return ktop ? ((ktop - 1) / SAMSIM_GB) * SAMSIM_GB + 1 : Na;
}

__device__ __noinline__ void grav_drain(Col& c, bool exact_all) {
  const View v = c;
  const int Na = c.N_active, N = CFG.Nlayer;
  const double dt = CFG.dt;
  Lay q = v.w1(), smin = v.w2(), fl_m = v.fl_m();
  double heat_loss = 0.0;

  SAMSIM_LOOP
  for (int k = Na; k <= N - 1; k++) v.ray()[k] = 0.0;  // :98 ray = 0 (entries below N_active are overwritten next)
  const double bottom_h = v.thick()[Na] * v.psi_s()[Na] / psi_s_min;  // thick(N_active)*psi_s(N_active)/psi_s_min
  const double S_br_Na = v.S_br()[Na];
  // Layers K0..Na are evaluated below; layers 1..K0-1 are proven unable to drain by the bound pass (lean steps only)
  const int K0 = (!exact_all && CFG.harmonic_flag == 2 && CFG.n_bgc == 0) ? grav_drain_bound(c, bottom_h, S_br_Na) : 1;
  // :104-106 permeability, thick/perm, and the order-independent suffix minimum of perm(k:Na-1), one backward pass
  double perm_Na = 0.0;
  int kmin_cand = 0, ncand = 0;  // candidates: layers whose estimate can exceed ray_crit
  {
    double mn = 0.0, sq = 0.0, st = 0.0, st_below = 0.0, qb_est = 0.0;  // suffix sums for the estimate
    SAMSIM_LOOP
    for (int k = Na; k >= K0; k--) {
      if (k - SAMSIM_PF >= K0) { v.psi_l().prefetch(k - SAMSIM_PF); v.thick().prefetch(k - SAMSIM_PF); v.S_br().prefetch(k - SAMSIM_PF); }
      const double pk = 1e-17 * det_pow(1000.0 * fabs(v.psi_l()[k]), 3.10);
      if (k == Na) { perm_Na = pk; qb_est = bottom_h / pk; continue; }  // perm itself is not needed again
      const double thk = v.thick()[k];
      const double qk = thk / pk;
      q[k] = qk;
      mn = (k == Na - 1) ? pk : f_min(mn, pk);
      if (exact_all) {
        smin[k] = mn;
      } else {
        st_below = st;          // ~SUM(thick(k+1:Na-1))
        sq = sq + qk;           // ~SUM(thick/perm (k:Na-1))
        st = st + thk;          // ~SUM(thick(k:Na-1))
        double est;
        if (CFG.harmonic_flag == 1) {
          est = grav * rho_l * bbeta * (v.S_br()[k] - S_br_Na) * (st_below + bottom_h) * f_min(mn, perm_Na);
          smin[k] = mn;  // needed again by the exact evaluation of candidates
        } else {
          const double hp = (mn < 1e-14) ? 0.0 : (st + bottom_h) / (sq + qb_est);
          est = grav * rho_l * bbeta * (v.S_br()[k] - S_br_Na) * (st_below + bottom_h) * hp;
        }
        est = est / (kappa_l * mu);
        // exactly 0 where the reference's value is exactly 0 (hp == 0); negative estimates clip like :135
        // (harmonic_flag 2: a candidate has est > 0, hence mn >= 1e-14: its exact evaluation needs no smin)
        const double rest = (CFG.harmonic_flag == 2 && mn < 1e-14) ? 0.0 : f_max(est, 0.0);
        v.ray()[k] = rest;
        if (rest > ray_crit * (1.0 - 1e-10)) { kmin_cand = k; ncand++; }
      }
    }
  }
  const double qb = bottom_h / perm_Na;

  // blocks of GB layers, from the bottom block upwards; `carry_t` = SUM(thick(k0+GB : Na-1)) of the block below.
  // All layers when ray is observable (exact_all); otherwise, when several layers are candidates, the blocks from the
  // topmost candidate down: the candidates of a column sit together (the warm lower part of the ice), and their
  // forward sums share every load -- evaluating them one by one in the drain loop is O(candidates x depth).
  const bool blocked = exact_all || ncand >= 3;
  const int kstop = exact_all ? 1 : kmin_cand;   // evaluate the blocks that reach up to this layer
  int kexact_from = exact_all ? 1 : Na;          // ray(k) is exact for k >= kexact_from
  double carry_t = 0.0;
  for (int k0 = ((Na - 2) / SAMSIM_GB) * SAMSIM_GB + 1; blocked && k0 >= 1 && k0 + SAMSIM_GB - 1 >= kstop && Na >= 2; k0 -= SAMSIM_GB) {
    kexact_from = k0;
    double aq[SAMSIM_GB], at[SAMSIM_GB];
#pragma unroll
    for (int j = 0; j < SAMSIM_GB; j++) { aq[j] = 0.0; at[j] = 0.0; }
    // The head and the per-layer evaluation below are rolled loops over register arrays (selects / a shift register):
    // unrolled they were 16 KB of straight-line code run three times per step, and the step kernel is bound by
    // instruction fetch as much as by anything else (profiles/README.md, round 2).
    SAMSIM_LOOP
    for (int d = 0; d < SAMSIM_GB; d++) {  // triangular head: layer k0+d feeds accumulators 0..d
      const int kk = k0 + d;
      if (kk <= Na - 1) {
        const double qv = q[kk], tv = v.thick()[kk];
#pragma unroll
        for (int j = 0; j < SAMSIM_GB; j++) {
          const double nq = aq[j] + qv, nt = at[j] + tv;
          aq[j] = (j <= d) ? nq : aq[j];
          at[j] = (j <= d) ? nt : at[j];
        }
      }
    }
    SAMSIM_LOOP
    for (int kk = k0 + SAMSIM_GB; kk <= Na - 1; kk++) {  // body: every accumulator takes every layer, in order
      // an iteration is 16 independent additions: the data must be requested several iterations ahead to arrive in time
      if (kk + 8 <= Na - 1) { q.prefetch(kk + 8); v.thick().prefetch(kk + 8); }
      const double qv = q[kk], tv = v.thick()[kk];
#pragma unroll
      for (int j = 0; j < SAMSIM_GB; j++) { aq[j] = aq[j] + qv; at[j] = at[j] + tv; }
    }
    const double carry_next = at[0];
    double below = carry_t;  // SUM(thick(k+1:Na-1)): the accumulator of the layer below (0 when there is none)
    SAMSIM_LOOP
    for (int j = SAMSIM_GB - 1; j >= 0; j--) {
      const int k = k0 + j;
      const double aqj = aq[SAMSIM_GB - 1], atj = at[SAMSIM_GB - 1];  // accumulators of layer k: top of the shift register
#pragma unroll
      for (int i = SAMSIM_GB - 1; i >= 1; i--) { aq[i] = aq[i - 1]; at[i] = at[i - 1]; }
      if (k <= Na - 1) {
        const double height = below + bottom_h;  // :128
        const double d_S_br = v.S_br()[k] - S_br_Na;
        double r;
        if (CFG.harmonic_flag == 1) {
          r = grav * rho_l * bbeta * d_S_br * height * f_min(smin[k], perm_Na);  // MINVAL(perm(k:N_active))
        } else {
          // :112-113 minval(perm(k:Na-1)) < 1e-14 -> harmonic_perm = 0.  Without exact_all the suffix minimum was not
          // stored; there the estimate is exactly 0 iff the minimum is below 1e-14 or S_br(k) <= S_br(Na), and in both
          // cases ray(k) = MAX(.., 0) is exactly 0 as well (height, harmonic_perm > 0 otherwise): such layers keep their 0
          const bool zero = exact_all ? (smin[k] < 1e-14) : (v.ray()[k] == 0.0);
          double hp;
          if (zero) {
            hp = 0.0;
          } else {                // :115-120
            hp = aqj + qb;
            hp = (atj + bottom_h) / hp;
          }
          r = grav * rho_l * bbeta * d_S_br * height * hp;
        }
        r = r / (kappa_l * mu);
        v.ray()[k] = f_max(r, 0.0);
      }
      below = atj;
    }
    carry_t = carry_next;
  }

  // :141 / :173 grav_salt = grav_salt + SUM(S_abs) before the drain loop and - SUM(S_abs) after it: both are
  // forward sums over the layers the loop visits in the same order, so they are accumulated inside it.
  double sum_before = 0.0, sum_after = 0.0;
  double min_S = 1e300;  // minimum over the S_abs values this routine leaves behind (:198)
  int kfirst = 0;        // first draining layer: fl_m(1:kfirst) == 0

  // Layers 1..K0-1 cannot drain (and kfirst == 0 there): each leaves S_abs as it is, so both sums take the same
  // additions from 0.0 and get the same bits
  SAMSIM_LOOP
  for (int k = 1; k <= K0 - 1; k++) {
    if (k + SAMSIM_PF <= K0 - 1) v.S_abs().prefetch(k + SAMSIM_PF);
    const double Sk = v.S_abs()[k];
    sum_before = sum_before + Sk;
    min_S = f_min(min_S, Sk);
  }
  sum_after = sum_before;

  double run = 0.0;  // running sum = fl_up(kk) for every kk not yet clamped
  double sbk = v.S_br()[K0];
  SAMSIM_LOOP
  for (int k = K0; k <= Na - 1; k++) {  // :144-171
    if (k + SAMSIM_PF <= Na) {
      // psi_s and m are only read for layers above ray_crit: prefetching them for every layer was 16 B of DRAM
      // traffic per layer and step for nothing
      v.ray().prefetch(k + SAMSIM_PF); v.S_abs().prefetch(k + SAMSIM_PF); v.S_br().prefetch(k + SAMSIM_PF);
    }
    double rk = v.ray()[k];
    const double Sk = v.S_abs()[k];
    const double sbk1 = v.S_br()[k + 1];
    if (k < kexact_from && rk > ray_crit * (1.0 - 1e-10)) {
      // candidate: the reference's forward sums (:115-120, :128) for this layer only, then ray(k) as at :126-136
      double hq = 0.0, ht = 0.0, hb = 0.0;
      SAMSIM_LOOP
      for (int kk = k; kk <= Na - 1; kk++) {
        const double tv = v.thick()[kk];
        hq = hq + q[kk];
        ht = ht + tv;
        if (kk > k) hb = hb + tv;
      }
      const double height = hb + bottom_h;
      const double d_S_br = sbk - S_br_Na;
      double r;
      if (CFG.harmonic_flag == 1) {
        r = grav * rho_l * bbeta * d_S_br * height * f_min(smin[k], perm_Na);
      } else {
        double hp = hq + qb;  // the estimate was > 0, so minval(perm(k:Na-1)) >= 1e-14 (:112) holds
        hp = (ht + bottom_h) / hp;
        r = grav * rho_l * bbeta * d_S_br * height * hp;
      }
      r = r / (kappa_l * mu);
      rk = f_max(r, 0.0);
      v.ray()[k] = rk;
    }
    double up = run;
    double S_after = Sk;
    double fl_down_k = 0.0;
    sum_before = sum_before + Sk;
    // same && chain as :145, evaluated left to right: psi_s and m are only touched where ray exceeds ray_crit
    if (rk > ray_crit && v.psi_s()[k] > 0.001 && Sk / v.m()[k] > 0.1 && sbk > sbk1) {
      if (kfirst == 0) { kfirst = k; fl_m[k] = 0.0; EVT(c, EV_GRAV_DRAINED); }  // fl_m(kfirst) = fl_up(kfirst-1) = 0: first face read by mass_transfer
      const double plk = v.psi_l()[k], thk = v.thick()[k], Tk = v.T()[k];
      double flux = x_grav * (rk - ray_crit) * dt * thk;
      flux = f_min(flux, plk * rho_l * thk);
      fl_down_k = flux;
      double Snew = Sk - flux * sbk;
      v.S_abs()[k] = Snew;
      S_after = Snew;
      if (Snew < 0.0) { c.status = 21234; return; }
      SCV(c, SC_GRAV_TEMP) = SCV(c, SC_GRAV_TEMP) + flux * Tk;
      v.H_abs()[k] = v.H_abs()[k] - flux * c_l * Tk;
      heat_loss = heat_loss + flux * c_l * Tk;
      run = run + flux;
      up = f_min(run, plk * rho_l * thk);
    }
    if (CFG.n_bgc) {  // :178-183 (sic: column N_active+1 is assigned from column N_active), fl_down(k) = this layer's flux
      const double cellNa = (k == Na - 1) ? v.A(AR_FB_D)[k] : v.A(AR_FB_A)[k];
      v.A(AR_FB_O)[k] = cellNa + fl_down_k;
      v.A(AR_FB_U)[k] = v.A(AR_FB_U)[k] + up;
    }
    if (kfirst) fl_m[k + 1] = up;            // fl_m(2:N_active+1) = fl_up(1:N_active), :177 (zeros above kfirst are not stored)
    else min_S = f_min(min_S, Sk);           // layers above the first draining layer keep this value
    sum_after = sum_after + S_after;
    sbk = sbk1;
  }
  if (kfirst) fl_m[Na + 1] = run;
  if (CFG.n_bgc) v.A(AR_FB_U)[Na] = v.A(AR_FB_U)[Na] + run;  // fl_up(N_active)
  const double fl_up_Na = run;
  {
    const double S_Na = v.S_abs()[Na];  // layer N_active never drains; inactive layers hold 0
    sum_before = sum_before + S_Na;
    sum_after = sum_after + S_Na;
  }
  SCV(c, SC_GRAV_SALT) = SCV(c, SC_GRAV_SALT) + sum_before;  // :141
  SCV(c, SC_GRAV_SALT) = SCV(c, SC_GRAV_SALT) - sum_after;   // :173

  // :188 -- nothing moves above the first draining layer (fl_m(1:kfirst) == 0); without any drainage nothing moves
  if (kfirst) mass_transfer(c, fl_m, v.S_bu(), kfirst);

  SCV(c, SC_GRAV_DRAIN) = SCV(c, SC_GRAV_DRAIN) + run;  // :190 fl_m(N_active+1)
  if (CFG.grav_heat_flag == 2) v.H_abs()[Na] = v.H_abs()[Na] + heat_loss - fl_up_Na * c_l * SCV(c, SC_T_BOTTOM);  // :193-195
  // :198 MINVAL(S_abs) < 0: layers above kfirst kept the values scanned by the drain loop (min_S); the others
  // were rewritten by mass_transfer and are scanned here
  double mn = min_S;
  if (kfirst) for (int k = kfirst; k <= Na; k++) mn = f_min(mn, v.S_abs()[k]);
  else mn = f_min(mn, v.S_abs()[Na]);
  if (f_min(mn, 0.0) < 0.0) c.status = 1337;  // (inactive layers are 0)
}

// fl_grav_drain_simple, mo_grav_drain.f90:218-279 (grav_flag 3)
__device__ __noinline__ void grav_drain_simple(Col& c) {
  const View v = c;
  const int Na = c.N_active, N = CFG.Nlayer;
  Lay perm = v.w0(), hperm = v.w2();
  SAMSIM_LOOP
  for (int k = 1; k <= N - 1; k++) v.ray()[k] = 0.0;
  SAMSIM_LOOP
  for (int k = 1; k <= Na; k++) perm[k] = 1e-17 * det_pow(1000.0 * fabs(v.psi_l()[k]), 3.10);
  const double bottom_h = v.thick()[Na] * v.psi_s()[Na] / psi_s_min;
  if (CFG.harmonic_flag == 2) {
    SAMSIM_LOOP
    for (int k = 1; k <= Na - 1; k++) {
      double mn = perm[k];
      SAMSIM_LOOP
      for (int kk = k; kk <= Na - 1; kk++) mn = f_min(mn, perm[kk]);
      if (mn < 1e-14) {
        hperm[k] = 0.0;
      } else {
        double h = 0.0;
        SAMSIM_LOOP
        for (int kk = k; kk <= Na - 1; kk++) h = h + v.thick()[kk] / perm[kk];
        h = h + bottom_h / perm[Na];
        hperm[k] = (sum_fwd(v.thick(), k, Na - 1) + bottom_h) / h;
      }
    }
  }
  const double S_br_Na = v.S_br()[Na];
  SAMSIM_LOOP
  for (int k = 1; k <= Na - 1; k++) {
    double d_S_br = v.S_br()[k] - S_br_Na;
    double height = sum_fwd(v.thick(), k + 1, Na - 1) + bottom_h;
    double r;
    if (CFG.harmonic_flag == 1) {
      double mn = perm[k];
      SAMSIM_LOOP
      for (int kk = k; kk <= Na; kk++) mn = f_min(mn, perm[kk]);
      r = grav * rho_l * bbeta * d_S_br * height * mn;
    } else {
      r = grav * rho_l * bbeta * d_S_br * height * hperm[k];
    }
    r = r / (kappa_l * mu);
    v.ray()[k] = f_max(r, 0.0);
  }
  SAMSIM_LOOP
  for (int k = Na - 1; k >= 1; k--)
    if (v.ray()[k] > ray_crit) v.S_abs()[k] = v.S_abs()[k] * SAMSIM_F32(0.99);
  SCV(c, SC_GRAV_DRAIN) = 0.0;
}

// ==========================================================================================
// mo_flood.f90
// ==========================================================================================

// flood, mo_flood.f90:55-153
__device__ __noinline__ void flood(Col& c) {
  const View v = c;
  const int Na = c.N_active;
  const double dt = CFG.dt, freeboard = SCV(c, SC_FREEBOARD), psi_g_snow = SCV(c, SC_PSI_G_SNOW);
  double& thick_snow = SCV(c, SC_THICK_SNOW);
  double& H_abs_snow = SCV(c, SC_H_ABS_SNOW);
  double& m_snow = SCV(c, SC_M_SNOW);
  double hp = 0.0;
  EVT(c, EV_FLOOD);
  SAMSIM_LOOP
  for (int k = 1; k <= Na - 1; k++) hp = hp + v.thick()[k] / (1e-17 * det_pow(1000.0 * v.psi_l()[k], 3.10));  // :73-79
  const double bottom_h = v.thick()[Na] * v.psi_s()[Na] / psi_s_min;
  hp = hp + bottom_h / (1e-17 * det_pow(1000.0 * v.psi_l()[Na], 3.10));
  hp = (sum_fwd(v.thick(), 1, Na - 1) + bottom_h) / hp;

  double flood_brine = -dt * grav * rho_l * rho_l * hp * (freeboard) / (mu * sum_fwd(v.thick(), 1, Na));  // :85
  const double shift_ice = flood_brine / (rho_l * psi_g_snow / ratio_flood);
  const double shift_snow = shift_ice * (1 + psi_g_snow / (1.0 - psi_g_snow) * (1.0 - 1.0 / ratio_flood));

  const double S_bu_Na = v.S_abs()[Na] / v.m()[Na];  // S_bu(k) = S_abs(k)/m(k) before any change, :93-95
  double S1 = v.S_abs()[1], H1 = v.H_abs()[1], m1 = v.m()[1], th1 = v.thick()[1];
  S1 = S1 + flood_brine * S_bu_Na;                  // :102-104
  H1 = H1 + flood_brine * v.H_abs()[Na] / v.m()[Na];
  m1 = m1 + flood_brine;
  th1 = th1 + shift_ice;                            // :107-112
  H1 = H1 + shift_snow / thick_snow * H_abs_snow;
  H_abs_snow = H_abs_snow - shift_snow / thick_snow * H_abs_snow;
  m1 = m1 + shift_snow / thick_snow * m_snow;
  m_snow = m_snow - shift_snow / thick_snow * m_snow;
  thick_snow = thick_snow - shift_snow;
  v.S_abs()[1] = S1; v.H_abs()[1] = H1; v.m()[1] = m1; v.thick()[1] = th1;  // Na > 1 here, layer 1 != layer Na

  if (freeboard + shift_ice < neg_free) {  // :117-138
    EVT(c, EV_FLOOD_NEG_FREE);
    const double shift = neg_free - (freeboard + shift_ice);
    flood_brine = shift * (psi_g_snow)*rho_l;
    const double T_Na = v.T()[Na];
    v.S_abs()[Na] = v.S_abs()[Na] + (SCV(c, SC_S_BU_BOTTOM) - S_bu_Na) * flood_brine;
    v.H_abs()[Na] = v.H_abs()[Na] + (SCV(c, SC_T_BOTTOM) - T_Na) * c_l * flood_brine;
    S1 = S1 + S_bu_Na * flood_brine;
    H1 = H1 + T_Na * c_l * flood_brine;
    m1 = m1 + flood_brine;
    th1 = th1 + shift;
    H1 = H1 + shift / thick_snow * H_abs_snow;
    H_abs_snow = H_abs_snow - shift / thick_snow * H_abs_snow;
    m1 = m1 + shift / thick_snow * m_snow;
    m_snow = m_snow - shift / thick_snow * m_snow;
    thick_snow = thick_snow - shift;
    v.S_abs()[1] = S1; v.H_abs()[1] = H1; v.m()[1] = m1; v.thick()[1] = th1;
  }
  if (CFG.n_bgc) {  // :140-144 fl_brine_bgc(N_active,1) and (N_active+1,N_active) += flood_brine
    Lay U = v.A(AR_FB_U);
    if (Na >= 3) c.fb_x = c.fb_x + flood_brine; else U[1] = U[1] + flood_brine;
    U[Na] = U[Na] + flood_brine;
  }
}

// flood_simple, mo_flood.f90:167-210
__device__ __forceinline__ void flood_simple(Col& c) {
  const View v = c;
  double& thick_snow = SCV(c, SC_THICK_SNOW);
  double& H_abs_snow = SCV(c, SC_H_ABS_SNOW);
  double& m_snow = SCV(c, SC_M_SNOW);
  const double shift = SCV(c, SC_FREEBOARD) - neg_free;
  const double flood_brine = -shift * SCV(c, SC_PSI_G_SNOW) * rho_l;
  EVT(c, EV_FLOOD_SIMPLE);
  double S1 = v.S_abs()[1], H1 = v.H_abs()[1], m1 = v.m()[1];
  v.thick()[1] = v.thick()[1] - shift;
  S1 = S1 + SCV(c, SC_S_BU_BOTTOM) * flood_brine;
  H1 = H1 - shift / thick_snow * H_abs_snow;
  H1 = H1 + SCV(c, SC_T_BOTTOM) * c_l * flood_brine;
  m1 = m1 - shift / thick_snow * m_snow;
  m1 = m1 + flood_brine;
  H_abs_snow = H_abs_snow + shift / thick_snow * H_abs_snow;
  m_snow = m_snow + shift / thick_snow * m_snow;
  thick_snow = thick_snow + shift;
  v.S_abs()[1] = S1; v.H_abs()[1] = H1; v.m()[1] = m1;
}

// ==========================================================================================
// mo_flush.f90
// ==========================================================================================

// flush3, mo_flush.f90:70-237.  Scratch: w0 R_v, w1 R_h, w2 R, w3 S_bu(local), fl_m.
__device__ __noinline__ void flush3(Col& c) {
  const View v = c;
  const int Na = c.N_active, N = CFG.Nlayer;
  const double dt = CFG.dt, freeboard = SCV(c, SC_FREEBOARD);
  Lay R_v = v.w0(), R_h = v.w1(), R = v.w2(), S_bu = v.w3(), fl_m = v.fl_m();
  double& melt_thick = SCV(c, SC_MELT_THICK);
  EVT(c, EV_FLUSH3);

  SAMSIM_LOOP
  for (int k = 1; k <= Na; k++) { v.flush_v()[k] = 0.0; v.flush_h()[k] = 0.0; }   // :101-102 (dummies are DIMENSION(N_active))
  SAMSIM_LOOP
  for (int k = 1; k <= Na; k++) S_bu[k] = v.S_abs()[k] / v.m()[k];              // :103
  const double konst = sum_fwd(v.thick(), 1, Na) * para_flush_horiz;          // :106
  melt_thick = f_min(melt_thick, v.psi_l()[1] * v.thick()[1]);                  // :110
  melt_thick = f_min(melt_thick, CFG.thick_0 / 3.0);                          // :112

  if (CFG.snow_flush_flag == 1) {  // :114-125
    SAMSIM_LOOP
    for (int k = Na + 1; k <= N; k++) v.perm()[k] = 0.0;
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) {
      double p = 1e-17 * det_pow(1000.0 * fabs(v.psi_l()[k] + 2. * v.psi_g()[k]), 3.10);
      if (p == 0.0) p = 1.0;
      v.perm()[k] = p;
    }
  } else if (CFG.snow_flush_flag == 0) {  // :126-130
    SAMSIM_LOOP
    for (int k = Na + 1; k <= N; k++) v.perm()[k] = 1.0;
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) v.perm()[k] = 1e-17 * det_pow(1000.0 * fabs(v.psi_l()[k]), 3.10);
  }
  SAMSIM_LOOP
  for (int k = 1; k <= Na; k++) {  // :133-137
    const double pk = f_max(v.perm()[k], 0.00000000000000000000001), thk = v.thick()[k];
    R_v[k] = mu * thk / pk;
    R_h[k] = mu * konst / (thk * pk);
  }
  R[Na] = 0.0;
  R[Na - 1] = R_v[Na - 1];
  SAMSIM_LOOP
  for (int k = Na - 2; k >= 1; k--) {  // :141-146
    double r = R[k + 1] + R_v[k];
    R[k] = ((r)*R_h[k]) / (r + R_h[k]);
  }
  const double T1 = v.T()[1];
  double flush_total = (freeboard + melt_thick) / R[1] * grav * dt * density_of(T1, S_br_of(T1)) * rho_l;  // :152
  flush_total = f_min(flush_total, melt_thick * rho_l);
  SCV(c, SC_MELT_ERR) = SCV(c, SC_MELT_ERR) + melt_thick - f_min(flush_total / rho_l, melt_thick);  // :156

  {
    const double den = R[2] + R_v[1] + R_h[1];
    v.flush_h()[1] = flush_total * (R[2] + R_v[1]) / den;  // :159-160
    v.flush_v()[1] = flush_total * R_h[1] / den;
  }
  SAMSIM_LOOP
  for (int k = 2; k <= Na - 1; k++) {  // :161-164
    const double fv = v.flush_v()[k - 1], a = R[k + 1] + R_v[k], den = a + R_h[k];
    v.flush_h()[k] = fv * a / den;
    v.flush_v()[k] = fv * R_h[k] / den;
  }
  v.flush_v()[Na] = v.flush_v()[Na - 1];
  v.flush_h()[Na] = 0.0;

  if (CFG.n_bgc) {  // :168-175
    Lay D = v.A(AR_FB_D), Ac = v.A(AR_FB_A);
    double sum_h = 0.0;
    SAMSIM_LOOP
    for (int k = 1; k <= Na - 1; k++) {
      const double fh = v.flush_h()[k];
      if (k == Na - 1) D[k] = D[k] + fh; else Ac[k] = Ac[k] + fh;  // cell (N_active-1, N_active) is the down-cell
      sum_h = sum_h + fh;
    }
    sum_h = sum_h + v.flush_h()[Na];
    D[Na] = D[Na] + sum_h;
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) D[k] = D[k] + v.flush_v()[k];
  }

  fl_m[1] = 0.0;  // :179-180
  SAMSIM_LOOP
  for (int k = 1; k <= Na; k++) fl_m[k + 1] = -v.flush_v()[k];

  mass_transfer(c, fl_m, S_bu);  // with the LOCAL S_bu (:182)
  const double T_Na = v.T()[Na];
  if (CFG.flush_heat_flag == 2) v.H_abs()[Na] = v.H_abs()[Na] - fl_m[Na + 1] * T_Na * c_l;  // :185-187

  v.m()[1] = v.m()[1] - flush_total;  // :190-191
  v.thick()[1] = v.thick()[1] - flush_total / rho_l;

  double sfh = 0.0;
  double H_Na = v.H_abs()[Na], S_Na = v.S_abs()[Na];
  SAMSIM_LOOP
  for (int k = 1; k <= Na - 1; k++) {  // :196-206
    const double fh = v.flush_h()[k], Tk = v.T()[k];
    const double loss_S = fh * S_br_of(Tk, v.S_abs()[k] / v.m()[k]);
    const double loss_H = fh * Tk * c_l;
    v.S_abs()[k] = v.S_abs()[k] - loss_S;
    v.H_abs()[k] = v.H_abs()[k] - loss_H;
    H_Na = H_Na + loss_H;
    S_Na = S_Na + loss_S;
    sfh = sfh + fh;
  }
  sfh = sfh + v.flush_h()[Na];  // SUM(flush_h) over the N_active-long dummy
  const double loss_S = sfh * S_bu[Na];  // :207-208
  const double loss_H = sfh * T_Na * c_l;
  if (CFG.flush_heat_flag == 2) H_Na = H_Na - loss_H;
  S_Na = S_Na - loss_S;
  v.H_abs()[Na] = H_Na;
  v.S_abs()[Na] = S_Na;

  double mn = v.S_abs()[1];
  SAMSIM_LOOP
  for (int k = 2; k <= Na; k++) mn = f_min(mn, v.S_abs()[k]);
  mn = f_min(mn, 0.0);  // MINVAL over all Nlayer: inactive layers hold 0 (only matters when Na < N)
  if (mn < -0.00000000000000000000000001) {
    EVT(c, EV_FLUSH3_CLAMP);
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) v.S_abs()[k] = f_max(v.S_abs()[k], 0.0);
  }
  if (fabs(v.m()[1]) < 0.000001) c.status = 9876;  // :230-233
}

// flush3 without tracers, with its sweeps merged (the melt season is bound by DRAM traffic: 109 KB per column-step at
// SHEBA state 345, profiles/r2_ncu_step_kernel_state345.json).  Same expressions, same order as flush3 above; the
// differences are where values live:
//   * R_v, R_h (:133-137) are recomputed from perm and thick where they are used instead of being stored;
//   * the new flush_v / flush_h are ADDED to the accumulated arrays as they are produced -- the driver's
//     old = cur; cur = 0; flush3; cur = cur + old (mo_grotz.f90:697-701, :736-737) is cur + new, and IEEE addition
//     commutes -- so the two copy sweeps and the zeroing disappear (flush_h of this step is kept in w3 for :196-206);
//   * the local S_bu = S_abs/m (:103) is evaluated inside mass_transfer from the values it reads anyway
//     (S_abs(k+1) before layer k+1 is updated, the carried pre-update value of layer k, m is not modified);
//   * fl_m (:179-180) is written by the flush_v sweep; the MINVAL of :218 rides along the horizontal-loss sweep.
// Scratch: w2 R, w3 flush_h of this step, fl_m.
__device__ __noinline__ void flush3_fused(Col& c) {
  const View v = c;
  const int Na = c.N_active, N = CFG.Nlayer;
  const double dt = CFG.dt, freeboard = SCV(c, SC_FREEBOARD);
  Lay R = v.w2(), fh_new = v.w3(), fl_m = v.fl_m();
  double& melt_thick = SCV(c, SC_MELT_THICK);
  EVT(c, EV_FLUSH3);

  const double konst = sum_fwd(v.thick(), 1, Na) * para_flush_horiz;          // :106
  melt_thick = f_min(melt_thick, v.psi_l()[1] * v.thick()[1]);                  // :110
  melt_thick = f_min(melt_thick, CFG.thick_0 / 3.0);                          // :112

  // :114-130 permeability (a state array: dat_perm), then :137-146 the resistance recurrence, one backward sweep
  if (CFG.snow_flush_flag == 1) {
    SAMSIM_LOOP
    for (int k = Na + 1; k <= N; k++) v.perm()[k] = 0.0;
  } else if (CFG.snow_flush_flag == 0) {
    SAMSIM_LOOP
    for (int k = Na + 1; k <= N; k++) v.perm()[k] = 1.0;
  }
  auto perm_of = [&](int k) {
    double p;
    if (CFG.snow_flush_flag == 1) {
      p = 1e-17 * det_pow(1000.0 * fabs(v.psi_l()[k] + 2. * v.psi_g()[k]), 3.10);
      if (p == 0.0) p = 1.0;
    } else {
      p = 1e-17 * det_pow(1000.0 * fabs(v.psi_l()[k]), 3.10);
    }
    return p;
  };
  double Rv1 = 0.0, Rh1 = 0.0, R2 = 0.0, R1 = 0.0;
  {
    double Rk1 = 0.0;  // R(k+1)
    SAMSIM_LOOP
    for (int k = Na; k >= 1; k--) {
      const double p = perm_of(k);
      v.perm()[k] = p;
      const double pk = f_max(p, 0.00000000000000000000001), thk = v.thick()[k];
      const double Rv = mu * thk / pk;
      const double Rh = mu * konst / (thk * pk);
      double Rk;
      if (k == Na) Rk = 0.0;                 // :138
      else if (k == Na - 1) Rk = Rv;         // :139
      else {                                 // :141-146
        const double r = Rk1 + Rv;
        Rk = ((r)*Rh) / (r + Rh);
      }
      R[k] = Rk;
      if (k == 2) R2 = Rk;
      if (k == 1) { R1 = Rk; Rv1 = Rv; Rh1 = Rh; }
      Rk1 = Rk;
    }
  }
  const double T1 = v.T()[1];
  double flush_total = (freeboard + melt_thick) / R1 * grav * dt * density_of(T1, S_br_of(T1)) * rho_l;  // :152
  flush_total = f_min(flush_total, melt_thick * rho_l);
  SCV(c, SC_MELT_ERR) = SCV(c, SC_MELT_ERR) + melt_thick - f_min(flush_total / rho_l, melt_thick);  // :156

  // :158-165 flush_h / flush_v top -> bottom, accumulated into the output arrays; fl_m(k+1) = -flush_v(k) (:179-180)
  fl_m[1] = 0.0;
  double sfh = 0.0;  // SUM(flush_h), forward
  {
    const double den = R2 + Rv1 + Rh1;
    double fh = flush_total * (R2 + Rv1) / den;   // :159-160
    double fv = flush_total * Rh1 / den;
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) {
      if (k >= 2 && k <= Na - 1) {                // :161-164
        const double pk = f_max(v.perm()[k], 0.00000000000000000000001), thk = v.thick()[k];
        const double Rv = mu * thk / pk;
        const double Rh = mu * konst / (thk * pk);
        const double a = R[k + 1] + Rv, den2 = a + Rh;
        fh = fv * a / den2;
        fv = fv * Rh / den2;
      } else if (k == Na) {
        fh = 0.0;                                  // flush_h(Na) = 0, flush_v(Na) = flush_v(Na-1)
      }
      v.flush_h()[k] = fh + v.flush_h()[k];
      v.flush_v()[k] = fv + v.flush_v()[k];
      fh_new[k] = fh;
      fl_m[k + 1] = -fv;
      if (k <= Na - 1) sfh = sfh + fh;
    }
  }
  const double fv_Na = -fl_m[Na + 1];

  // :182 mass_transfer with the LOCAL S_bu = S_abs/m of the state before the transfer (mo_mass.f90:53-96)
  const double T_bottom = SCV(c, SC_T_BOTTOM), S_bu_bottom = SCV(c, SC_S_BU_BOTTOM);
  double sbu_Na;
  {
    double T_km1 = 0.0, Sbu_km1 = 0.0, Sabs_km1 = 0.0;
    double T_k = v.T()[1], Sbu_k = v.S_abs()[1] / v.m()[1];
    double f0 = 0.0;
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) {
      double T_kp1, Sbu_kp1, Sabs_kp1;
      if (k < Na) {
        T_kp1 = v.T()[k + 1];
        Sabs_kp1 = v.S_abs()[k + 1];
        Sbu_kp1 = Sabs_kp1 / v.m()[k + 1];
      } else {
        T_kp1 = T_bottom; Sbu_kp1 = S_bu_bottom; Sabs_kp1 = S_bu_bottom * 2000.0;
      }
      const double f1 = fl_m[k + 1];
      double H = v.H_abs()[k], S = v.S_abs()[k];
      mass_transfer_layer(f1, f0, T_km1, Sbu_km1, Sabs_km1, T_k, Sbu_k, T_kp1, Sbu_kp1, Sabs_kp1, H, S);
      v.H_abs()[k] = H;
      v.S_abs()[k] = S;
      T_km1 = T_k; Sbu_km1 = Sbu_k; Sabs_km1 = S;
      if (k < Na) { T_k = T_kp1; Sbu_k = Sbu_kp1; }
      f0 = f1;
    }
    sbu_Na = Sbu_k;  // S_bu(N_active) of :103
  }
  const double T_Na = v.T()[Na];
  if (CFG.flush_heat_flag == 2) v.H_abs()[Na] = v.H_abs()[Na] - (-fv_Na) * T_Na * c_l;  // :185-187 (fl_m(Na+1) = -flush_v(Na))

  v.m()[1] = v.m()[1] - flush_total;  // :190-191
  v.thick()[1] = v.thick()[1] - flush_total / rho_l;

  double H_Na = v.H_abs()[Na], S_Na = v.S_abs()[Na];
  double mn = 1e300;
  SAMSIM_LOOP
  for (int k = 1; k <= Na - 1; k++) {  // :196-206
    const double fh = fh_new[k], Tk = v.T()[k];
    const double Sk = v.S_abs()[k];
    const double loss_S = fh * S_br_of(Tk, Sk / v.m()[k]);
    const double loss_H = fh * Tk * c_l;
    const double Snew = Sk - loss_S;
    v.S_abs()[k] = Snew;
    v.H_abs()[k] = v.H_abs()[k] - loss_H;
    H_Na = H_Na + loss_H;
    S_Na = S_Na + loss_S;
    mn = f_min(mn, Snew);
  }
  // SUM(flush_h) over the N_active-long dummy: sfh + flush_h(Na) = sfh + 0
  sfh = sfh + 0.0;
  const double loss_S = sfh * sbu_Na;  // :207-208
  const double loss_H = sfh * T_Na * c_l;
  if (CFG.flush_heat_flag == 2) H_Na = H_Na - loss_H;
  S_Na = S_Na - loss_S;
  v.H_abs()[Na] = H_Na;
  v.S_abs()[Na] = S_Na;
  mn = f_min(mn, S_Na);
  mn = f_min(mn, 0.0);  // MINVAL over all Nlayer: inactive layers hold 0
  if (mn < -0.00000000000000000000000001) {  // :218-227
    EVT(c, EV_FLUSH3_CLAMP);
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) v.S_abs()[k] = f_max(v.S_abs()[k], 0.0);
  }
  if (fabs(v.m()[1]) < 0.000001) c.status = 9876;  // :230-233
}

// flush4, mo_flush.f90:253-296 (flush_flag 6)
__device__ __noinline__ void flush4(Col& c) {
  const View v = c;
  const int N = CFG.Nlayer, Na = c.N_active;
  double& melt_thick = SCV(c, SC_MELT_THICK);
  const double S_bu1 = v.S_abs()[1] / v.m()[1], T1 = v.T()[1];
  EVT(c, EV_FLUSH4);
  v.H_abs()[1] = v.H_abs()[1] - melt_thick * rho_l * c_l * T1;
  v.S_abs()[1] = v.S_abs()[1] - melt_thick * rho_l * S_br_of(T1, S_bu1);
  v.thick()[1] = v.thick()[1] - melt_thick;
  v.m()[1] = v.m()[1] - melt_thick * rho_l;
  melt_thick = 0.0;
  int k = 2;
  while (k <= N && v.psi_l()[k] > v.psi_l()[k - 1]) {
    v.S_abs()[k] = para_flush_gamma * v.S_abs()[k];
    k = k + 1;
  }
  v.S_abs()[1] = f_max(v.S_abs()[1], 0.00);
  double mn = v.S_abs()[1];
  SAMSIM_LOOP
  for (int q = 2; q <= Na; q++) mn = f_min(mn, v.S_abs()[q]);
  if (mn < 0.0) c.status = 9876;
}

// ==========================================================================================
// mo_layer_dynamics.f90.  Snapshots rho/S_bu/H of the reference become w0/w1/w2.
// ==========================================================================================
__device__ __forceinline__ void snapshot_layers(Col& c, int k0, int k1) {
  const View v = c;
  SAMSIM_LOOP
  for (int k = k0; k <= k1; k++) {
    const double mk = v.m()[k];
    v.w0()[k] = mk / v.thick()[k];   // rho
    v.w1()[k] = v.S_abs()[k] / mk;   // S_bu
    v.w2()[k] = v.H_abs()[k] / mk;   // H
  }
}

// top_melt, mo_layer_dynamics.f90:191-326
__device__ __noinline__ void top_melt(Col& c) {
  const View v = c;
  const int N = CFG.Nlayer, N_middle = CFG.N_middle, N_top = CFG.N_top;
  const double thick_0 = CFG.thick_0;
  Lay rho = v.w0(), S_bu = v.w1(), H = v.w2();
  snapshot_layers(c, 1, c.N_active);  // :218-223
  v.m()[1] = v.m()[1] + v.m()[2];           // :231-235
  v.S_abs()[1] = v.S_abs()[1] + v.S_abs()[2];
  v.H_abs()[1] = v.H_abs()[1] + v.H_abs()[2];
  v.thick()[1] = v.thick()[1] + v.thick()[2];
  const int kmax = (N_top - 1 < c.N_active - 1) ? N_top - 1 : c.N_active - 1;
  SAMSIM_LOOP
  for (int k = 2; k <= kmax; k++) {  // :238-243
    v.m()[k] = rho[k + 1] * thick_0;
    v.S_abs()[k] = S_bu[k + 1] * rho[k + 1] * thick_0;
    v.H_abs()[k] = H[k + 1] * rho[k + 1] * thick_0;
  }
  if (c.N_active <= N_top) {  // :247-254
    EVT(c, EV_TOP_MELT_A);
    const int Na = c.N_active;
    v.m()[Na] = 0.0; v.S_abs()[Na] = 0.0; v.H_abs()[Na] = 0.0; v.thick()[Na] = 0.0;
    c.N_active = Na - 1;
  } else if (c.N_active > N_top && c.N_active <= N && v.thick()[N_top + 1] / thick_0 < 1.00001) {  // :256-273
    EVT(c, EV_TOP_MELT_B);
    const int Na = c.N_active;
    SAMSIM_LOOP
    for (int k = N_top; k <= Na - 1; k++) {
      v.m()[k] = rho[k + 1] * thick_0;
      v.S_abs()[k] = S_bu[k + 1] * rho[k + 1] * thick_0;
      v.H_abs()[k] = H[k + 1] * rho[k + 1] * thick_0;
    }
    v.m()[Na] = 0.0; v.S_abs()[Na] = 0.0; v.H_abs()[Na] = 0.0; v.thick()[Na] = 0.0;
    c.N_active = Na - 1;
  }
  if (c.N_active == N && v.thick()[N_top + 1] - thick_0 >= 0.000001) {  // :275-314
    EVT(c, EV_TOP_MELT_C);
    double loss_m = thick_0 * rho[N_top + 1];
    double loss_S = loss_m * S_bu[N_top + 1];
    double loss_H = loss_m * H[N_top + 1];
    v.m()[N_top] = loss_m;
    v.S_abs()[N_top] = loss_S;
    v.H_abs()[N_top] = loss_H;
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= N_middle + N_top; k++) {
      double mk = v.m()[k] - loss_m, Hk = v.H_abs()[k] - loss_H, Sk = v.S_abs()[k] - loss_S;
      const double shift = thick_0 * (double)(float)(N_middle - k + N_top) / (double)(float)(N_middle);  // :293
      loss_m = shift * rho[k + 1];
      loss_S = loss_m * S_bu[k + 1];
      loss_H = loss_m * H[k + 1];
      v.m()[k] = mk + loss_m;
      v.H_abs()[k] = Hk + loss_H;
      v.S_abs()[k] = Sk + loss_S;
    }
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= N_top + N_middle; k++) v.thick()[k] = v.thick()[k] - thick_0 / (double)(float)(N_middle);
  }
  // :318-321 grid consistency, STOP 7889 (SUM(thick) over all layers; inactive are 0)
  if (c.N_active < N) {
    if (thick_0 * (c.N_active + 0.501) <= sum_fwd(v.thick(), 1, N)) c.status = 7889;
  }
}

// bottom_melt, mo_layer_dynamics.f90:341-420
__device__ __noinline__ void bottom_melt(Col& c) {
  const View v = c;
  const int N = CFG.Nlayer, N_middle = CFG.N_middle, N_top = CFG.N_top;
  Lay rho = v.w0(), S_bu = v.w1(), H = v.w2();
  snapshot_layers(c, N_top + 1, N);  // :364-370
  const double thN = v.thick()[N];
  double loss_m = 0.0, loss_S = 0.0, loss_H = 0.0;
  SAMSIM_LOOP
  for (int k = N_top + 1; k <= N_top + N_middle; k++) {  // :378-400
    double mk = v.m()[k] + loss_m, Hk = v.H_abs()[k] + loss_H, Sk = v.S_abs()[k] + loss_S;
    const double shift = thN * (k - N_top) / (double)(float)(N_middle);
    loss_m = shift * rho[k];
    loss_H = loss_m * H[k];
    loss_S = loss_m * S_bu[k];
    v.m()[k] = mk - loss_m;
    v.H_abs()[k] = Hk - loss_H;
    v.S_abs()[k] = Sk - loss_S;
  }
  SAMSIM_LOOP
  for (int k = N_top + 1; k <= N_top + N_middle; k++) v.thick()[k] = v.thick()[k] - thN / (double)(float)(N_middle);
  SAMSIM_LOOP
  for (int k = N_top + N_middle + 1; k <= N; k++) {  // :410-415
    const double thk = v.thick()[k];
    v.H_abs()[k] = rho[k - 1] * thk * H[k - 1];
    v.S_abs()[k] = rho[k - 1] * thk * S_bu[k - 1];
    v.m()[k] = rho[k - 1] * thk;
  }
}

// bottom_growth, mo_layer_dynamics.f90:438-520
__device__ __noinline__ void bottom_growth(Col& c) {
  const View v = c;
  const int N = CFG.Nlayer, N_middle = CFG.N_middle, N_top = CFG.N_top, N_bottom = CFG.N_bottom;
  Lay rho = v.w0(), S_bu = v.w1(), H = v.w2();
  snapshot_layers(c, N_top + 1, N_top + N_middle + 1);  // :463-468
  const double thN = v.thick()[N];
  double gain_m = 0.0, gain_S = 0.0, gain_H = 0.0;
  SAMSIM_LOOP
  for (int k = N_top + 1; k <= N_top + N_middle; k++) {  // :476-495
    double mk = v.m()[k] - gain_m, Hk = v.H_abs()[k] - gain_H, Sk = v.S_abs()[k] - gain_S;
    const double shift = thN * (k - N_top) / (double)(float)(N_middle);
    gain_m = shift * rho[k + 1];
    gain_H = gain_m * H[k + 1];
    gain_S = gain_m * S_bu[k + 1];
    v.m()[k] = mk + gain_m;
    v.H_abs()[k] = Hk + gain_H;
    v.S_abs()[k] = Sk + gain_S;
  }
  SAMSIM_LOOP
  for (int k = N_top + 1; k <= N_top + N_middle; k++) v.thick()[k] = v.thick()[k] + thN / (double)(float)(N_middle);
  SAMSIM_LOOP
  for (int k = N - N_bottom + 1; k <= N - 1; k++) {  // :503-508
    v.H_abs()[k] = v.H_abs()[k + 1];
    v.S_abs()[k] = v.S_abs()[k + 1];
    v.m()[k] = v.m()[k + 1];
  }
  const double mN = v.thick()[N] * rho_l;  // :511-513
  v.m()[N] = mN;
  v.H_abs()[N] = mN * SCV(c, SC_T_BOTTOM) * c_l;
  v.S_abs()[N] = mN * SCV(c, SC_S_BU_BOTTOM);
}

// bottom_growth_simple :537-561, bottom_melt_simple :573-590
__device__ __forceinline__ void bottom_growth_simple(Col& c) {
  const View v = c;
  const int Na = c.N_active + 1;
  c.N_active = Na;
  v.thick()[Na] = CFG.thick_0;
  const double mN = CFG.thick_0 * rho_l;
  v.m()[Na] = mN;
  v.H_abs()[Na] = mN * SCV(c, SC_T_BOTTOM) * c_l;
  v.S_abs()[Na] = mN * SCV(c, SC_S_BU_BOTTOM);
}
__device__ __forceinline__ void bottom_melt_simple(Col& c) {
  const View v = c;
  const int Na = c.N_active;
  v.thick()[Na] = 0.0; v.m()[Na] = 0.0; v.S_abs()[Na] = 0.0; v.H_abs()[Na] = 0.0;
  c.N_active = Na - 1;
}

// top_grow, mo_layer_dynamics.f90:607-716
__device__ __noinline__ void top_grow(Col& c) {
  const View v = c;
  const int N = CFG.Nlayer, N_middle = CFG.N_middle, N_top = CFG.N_top;
  const double thick_0 = CFG.thick_0;
  Lay rho = v.w0(), S_bu = v.w1(), H = v.w2();
  snapshot_layers(c, 1, c.N_active);  // :631-636
  {
    const double loss_m = thick_0 * rho[1];  // :639-648
    const double loss_S = loss_m * S_bu[1];
    const double loss_H = loss_m * H[1];
    v.m()[1] = v.m()[1] - loss_m;
    v.S_abs()[1] = v.S_abs()[1] - loss_S;
    v.H_abs()[1] = v.H_abs()[1] - loss_H;
    v.thick()[1] = v.thick()[1] - thick_0;
  }
  const int kmax = (N_top < c.N_active) ? N_top : c.N_active;
  SAMSIM_LOOP
  for (int k = 2; k <= kmax; k++) {  // :651-656
    v.m()[k] = rho[k - 1] * thick_0;
    v.S_abs()[k] = S_bu[k - 1] * rho[k - 1] * thick_0;
    v.H_abs()[k] = H[k - 1] * rho[k - 1] * thick_0;
  }
  if (c.N_active <= N_top) {  // :659-665
    EVT(c, EV_TOP_GROW_A);
    const int Na = c.N_active + 1;
    c.N_active = Na;
    v.m()[Na] = rho[Na - 1] * thick_0;
    v.S_abs()[Na] = S_bu[Na - 1] * thick_0 * rho[Na - 1];
    v.H_abs()[Na] = H[Na - 1] * thick_0 * rho[Na - 1];
    v.thick()[Na] = thick_0;
  } else if (c.N_active > N_top && c.N_active < N) {  // :668-680
    EVT(c, EV_TOP_GROW_B);
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= c.N_active; k++) {
      v.m()[k] = rho[k - 1] * thick_0;
      v.S_abs()[k] = S_bu[k - 1] * rho[k - 1] * thick_0;
      v.H_abs()[k] = H[k - 1] * rho[k - 1] * thick_0;
    }
    const int Na = c.N_active + 1;
    c.N_active = Na;
    v.m()[Na] = rho[Na - 1] * thick_0;
    v.S_abs()[Na] = S_bu[Na - 1] * thick_0 * rho[Na - 1];
    v.H_abs()[Na] = H[Na - 1] * thick_0 * rho[Na - 1];
    v.thick()[Na] = thick_0;
  } else if (c.N_active == N) {  // :682-711
    EVT(c, EV_TOP_GROW_C);
    double loss_m = thick_0 * rho[N_top];
    double loss_S = loss_m * S_bu[N_top];
    double loss_H = loss_m * H[N_top];
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= N_middle + N_top; k++) {
      double mk = v.m()[k] + loss_m, Hk = v.H_abs()[k] + loss_H, Sk = v.S_abs()[k] + loss_S;
      const double shift = thick_0 * (double)(float)(N_middle - k + N_top) / (double)(float)(N_middle);
      loss_m = shift * rho[k];
      loss_S = loss_m * S_bu[k];
      loss_H = loss_m * H[k];
      v.m()[k] = mk - loss_m;
      v.H_abs()[k] = Hk - loss_H;
      v.S_abs()[k] = Sk - loss_S;
    }
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= N_top + N_middle; k++) v.thick()[k] = v.thick()[k] + thick_0 / (double)(float)(N_middle);
  }
}


// ==========================================================================================
// Passive tracers (bgc_flag 2): mo_mass.f90:150-209 and the bgc lines of mo_layer_dynamics.f90
// ==========================================================================================
//
// fl_brine_bgc is an (Nlayer+1)^2 matrix in the reference, but only these cells are ever written
// (Na = N_active, Na+1 = the ocean):
//   (k,k+1)  k = 1..Na    expulsion (mo_grotz.f90:316-320), flush_v (mo_flush.f90:171-173)        -> D[k]
//   (k+1,k)  k = 1..Na    fl_up of gravity drainage (mo_grav_drain.f90:181-183), flooding (Na+1,Na) -> U[k]
//   (k,Na)   k = 1..Na-2  flush_h (mo_flush.f90:169); for k = Na-1 this IS the cell (k,k+1) = D[k]    -> A[k]
//   (k,Na+1) k = 1..Na-1  fl_down of gravity drainage (:179); for k = Na it is the cell D[Na]         -> O[k]
//   (Na,1)                flooding (mo_flood.f90:141); for Na = 2 it is the cell U[1]                 -> fb_x
// The arrays are step-local: the S5 sweep assigns D and clears U, A, O, fb_x (the reference zeroes the matrix
// after bgc_advection, mo_grotz.f90:745).
__device__ __forceinline__ double fb_get(const Col& c, int Na, int i, int j) {
  const View v = c;
  if (j == i + 1 && i <= Na) return v.A(AR_FB_D)[i];
  if (i == j + 1 && j <= Na) return v.A(AR_FB_U)[j];
  if (j == Na && i <= Na - 2) return v.A(AR_FB_A)[i];
  if (j == Na + 1 && i <= Na - 1) return v.A(AR_FB_O)[i];
  if (i == Na && j == 1 && Na >= 3) return c.fb_x;
  return 0.0;
}

// bgc_advection.  The reference visits every (i,j) pair; an empty cell moves MIN(0*br, abs/3) = 0 and x -/+ 0 is x,
// so rows whose content is non-negative (and whose brine concentration is finite) only visit their written cells,
// in the same ascending-j order; any other row runs the dense loop.  temp/br are the scratch arrays w0/w1.
__device__ __noinline__ void bgc_advection(Col& c) {
  const View v = c;
  const int Na = c.N_active;
  Lay temp = v.w0(), br = v.w1();
  Lay D = v.A(AR_FB_D), U = v.A(AR_FB_U), Ac = v.A(AR_FB_A), O = v.A(AR_FB_O);
  for (int q = 0; q < CFG.n_bgc; q++) {
    Lay x = v.bgc(q);
    const double bottom = SCV(c, SC_BGC_BOTTOM1 + q);
    // bgc_temp = bgc_abs (layers below N_active are not touched: copied back unchanged) and bgc_br, :171
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) {
      const double xk = x[k];
      temp[k] = xk;
      br[k] = xk / (f_max(v.psi_l()[k] * v.thick()[k] * rho_l, 0.000000000000001));
    }
    SAMSIM_LOOP
    for (int i = 1; i <= Na; i++) {  // :179-190
      const double xi = x[i], bi = br[i], lim = xi / 3.0;
      if (xi >= 0.0 && bi - bi == 0.0) {
        if (i == Na && Na >= 3) { const double f = f_min(c.fb_x * bi, lim); temp[i] = temp[i] - f; temp[1] = temp[1] + f; }
        if (i >= 2) { const double f = f_min(U[i - 1] * bi, lim); temp[i] = temp[i] - f; temp[i - 1] = temp[i - 1] + f; }
        if (i <= Na - 1) { const double f = f_min(D[i] * bi, lim); temp[i] = temp[i] - f; temp[i + 1] = temp[i + 1] + f; }
        if (i <= Na - 2) { const double f = f_min(Ac[i] * bi, lim); temp[i] = temp[i] - f; temp[Na] = temp[Na] + f; }
      } else {
        for (int j = 1; j <= Na; j++) {
          const double f = f_min(fb_get(c, Na, i, j) * bi, lim);
          temp[i] = temp[i] - f;
          temp[j] = temp[j] + f;
        }
      }
    }
    // :193-199 flows which leave the domain, then :202-208 flows which enter it -- only cell (Na+1, Na) is ever
    // written, the other layers receive 0*bgc_bottom = 0 -- and bgc_abs = bgc_temp
    SAMSIM_LOOP
    for (int i = 1; i <= Na; i++) {
      const double cell = (i == Na) ? D[i] : O[i];
      const double f = f_min(cell * br[i], x[i] / 3.0);
      double t = temp[i] - f;
      t = t + ((i == Na) ? U[Na] : 0.0) * bottom;
      x[i] = t;
    }
  }
}

// The six layer-dynamics routines treat a tracer exactly like S_abs (bgc_bulk = bgc/m next to S_bu = S_abs/m, the
// same products in the same order, bgc_bottom in the place of S_bu_bottom).  tracer_layer_dynamics replays the
// routine layer_dynamics() is about to run, for one tracer array, BEFORE m / thick / N_active change; rho and bulk
// are recomputed from that untouched state, so they equal the reference's snapshots.  `op` = routine chosen by the
// dispatcher below: 1 bottom_melt, 2 bottom_melt_simple, 3 bottom_growth_simple, 4 bottom_growth, 5 top_grow, 6 top_melt.
__device__ __noinline__ void tracer_layer_dynamics(Col& c, int op, Lay x, double bottom) {
  const View v = c;
  const int N = CFG.Nlayer, N_top = CFG.N_top, N_middle = CFG.N_middle, N_bottom = CFG.N_bottom, Na = c.N_active;
  const double thick_0 = CFG.thick_0;
  Lay bulk = v.w3();
  auto rho = [&](int k) { return v.m()[k] / v.thick()[k]; };
  if (op == 2) { x[Na] = 0.0; return; }                                             // bottom_melt_simple :586
  if (op == 3) { x[Na + 1] = bottom * (thick_0 * rho_l); return; }                  // bottom_growth_simple :557, m = thick_0*rho_l
  if (op == 1) {  // bottom_melt :341-420
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= N; k++) bulk[k] = x[k] / v.m()[k];
    double loss = 0.0;
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= N_top + N_middle; k++) {
      double xk = x[k] + loss;
      const double shift = v.thick()[N] * (k - N_top) / (double)(float)(N_middle);
      const double loss_m = shift * rho(k);
      loss = loss_m * bulk[k];
      x[k] = xk - loss;
    }
    // thick(k) of the bottom layers is not touched by the routine
    SAMSIM_LOOP
    for (int k = N_top + N_middle + 1; k <= N; k++) x[k] = rho(k - 1) * v.thick()[k] * bulk[k - 1];
    return;
  }
  if (op == 4) {  // bottom_growth :438-520
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= N_top + N_middle + 1; k++) bulk[k] = x[k] / v.m()[k];
    double gain = 0.0;
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= N_top + N_middle; k++) {
      double xk = x[k] - gain;
      const double shift = v.thick()[N] * (k - N_top) / (double)(float)(N_middle);
      const double gain_m = shift * rho(k + 1);
      gain = gain_m * bulk[k + 1];
      x[k] = xk + gain;
    }
    SAMSIM_LOOP
    for (int k = N - N_bottom + 1; k <= N - 1; k++) x[k] = x[k + 1];
    x[N] = (v.thick()[N] * rho_l) * bottom;  // m(Nlayer)*bgc_bottom with the new m(Nlayer) = thick(Nlayer)*rho_l
    return;
  }
  // top_grow / top_melt work on layers 1..N_active
  SAMSIM_LOOP
  for (int k = 1; k <= Na; k++) bulk[k] = x[k] / v.m()[k];
  if (op == 5) {  // top_grow :607-716
    {
      const double loss_m = thick_0 * rho(1);
      x[1] = x[1] - loss_m * bulk[1];
    }
    const int kmax = (N_top < Na) ? N_top : Na;
    SAMSIM_LOOP
    for (int k = 2; k <= kmax; k++) x[k] = bulk[k - 1] * rho(k - 1) * thick_0;
    if (Na <= N_top) {
      x[Na + 1] = bulk[Na] * thick_0 * rho(Na);
    } else if (Na > N_top && Na < N) {
      SAMSIM_LOOP
      for (int k = N_top + 1; k <= Na; k++) x[k] = bulk[k - 1] * rho(k - 1) * thick_0;
      x[Na + 1] = bulk[Na] * thick_0 * rho(Na);
    } else if (Na == N) {
      double loss_m = thick_0 * rho(N_top);
      double loss = loss_m * bulk[N_top];
      SAMSIM_LOOP
      for (int k = N_top + 1; k <= N_middle + N_top; k++) {
        const double xk = x[k] + loss;
        const double shift = thick_0 * (double)(float)(N_middle - k + N_top) / (double)(float)(N_middle);
        loss_m = shift * rho(k);
        loss = loss_m * bulk[k];
        x[k] = xk - loss;
      }
    }
    return;
  }
  // op == 6: top_melt :191-326
  x[1] = x[1] + x[2];
  {
    const int kmax = (N_top - 1 < Na - 1) ? N_top - 1 : Na - 1;
    SAMSIM_LOOP
    for (int k = 2; k <= kmax; k++) x[k] = bulk[k + 1] * rho(k + 1) * thick_0;
  }
  int Nb = Na;
  if (Na <= N_top) {
    x[Na] = 0.0;
    Nb = Na - 1;
  } else if (Na > N_top && Na <= N && v.thick()[N_top + 1] / thick_0 < 1.00001) {
    SAMSIM_LOOP
    for (int k = N_top; k <= Na - 1; k++) x[k] = bulk[k + 1] * rho(k + 1) * thick_0;
    x[Na] = 0.0;
    Nb = Na - 1;
  }
  if (Nb == N && v.thick()[N_top + 1] - thick_0 >= 0.000001) {
    double loss_m = thick_0 * rho(N_top + 1);
    double loss = loss_m * bulk[N_top + 1];
    x[N_top] = loss;
    SAMSIM_LOOP
    for (int k = N_top + 1; k <= N_middle + N_top; k++) {
      const double xk = x[k] - loss;
      const double shift = thick_0 * (double)(float)(N_middle - k + N_top) / (double)(float)(N_middle);
      loss_m = shift * rho(k + 1);
      loss = loss_m * bulk[k + 1];
      x[k] = xk + loss;
    }
  }
}

// layer_dynamics dispatcher, mo_layer_dynamics.f90:64-175 (SURVEY Appendix C)
__device__ __noinline__ void layer_dynamics(Col& c) {
  const View v = c;
  const int N = CFG.Nlayer, N_top = CFG.N_top, Na = c.N_active;
  const double thick_0 = CFG.thick_0;
  const bool bf = (CFG.bottom_flag == 1);
  const int nm1 = (Na - 1 > 1) ? Na - 1 : 1;
  const double phi_Na = v.phi()[Na], phi_nm1 = v.phi()[nm1], th1 = v.thick()[1];
  const double mid_ratio = v.thick()[N_top + 1] / thick_0;
  // tracers first (they read the untouched m, thick, N_active), then the routine itself
  auto tracers = [&](int op) {
    for (int q = 0; q < CFG.n_bgc; q++) tracer_layer_dynamics(c, op, v.bgc(q), SCV(c, SC_BGC_BOTTOM1 + q));
  };
  if (v.phi()[N - 1] <= psi_s_min / 2.0 && phi_Na < 0.00001 && Na == N && mid_ratio > 1.000001 && bf) {
    EVT(c, EV_BOTTOM_MELT);
    tracers(1);
    bottom_melt(c);
  } else if (Na > 1 && Na < N && phi_Na < 0.00001 && phi_nm1 <= psi_s_min / 2.0 && bf) {
    EVT(c, EV_BOTTOM_MELT_SIMPLE_A);
    tracers(2);
    bottom_melt_simple(c);
  } else if (Na > 1 && phi_Na < 0.00001 && phi_nm1 <= psi_s_min / 2.0 && mid_ratio < 1.01 && bf) {
    EVT(c, EV_BOTTOM_MELT_SIMPLE_B);
    tracers(2);
    bottom_melt_simple(c);
  } else if (phi_Na > psi_s_min && Na < N && bf) {
    EVT(c, EV_BOTTOM_GROWTH_SIMPLE);
    tracers(3);
    bottom_growth_simple(c);
  } else if (v.phi()[N] > psi_s_min && bf) {
    EVT(c, EV_BOTTOM_GROWTH);
    tracers(4);
    bottom_growth(c);
  } else if (th1 > 1.5 * thick_0) {
    SCV(c, SC_MTO3) = SCV(c, SC_MTO3) - th1;
    tracers(5);
    top_grow(c);
    SCV(c, SC_MTO3) = SCV(c, SC_MTO3) + v.thick()[1];
  } else if (th1 < 0.5 * thick_0) {
    SCV(c, SC_MTO3) = SCV(c, SC_MTO3) - th1;
    tracers(6);
    top_melt(c);
    SCV(c, SC_MTO3) = SCV(c, SC_MTO3) + v.thick()[1];
  }
}

}  // namespace samsim
