// step.cuh -- one iteration of the reference's time loop (mo_grotz.f90:182-835) for one column,
// plus the surface energy balance (mo_heat_fluxes.f90:69-312).  See physics.cuh for the
// arithmetic contract.
#pragma once

#include "physics.cuh"

namespace samsim {

// forcing tables visible to a thread
struct Forcing {
  // atmoflux_flag 2: window of records, [(site*4 + kind)*win_len + r]: staged in shared memory, or (global) the
  // whole table in global memory with win_len = nrec and win_first = 1
  const double* win;
  int win_len;            // records in the window
  int win_first;          // 1-based record number of window element 0
  int site;               // this column's site
  double scale[4], offset[4];  // kind order: fl_sw, fl_lw, T2m, precip
  // lab series in global memory, [(set*4 + kind)*nrec + r], kinds Tice, snowfall, heat, styropor
  const double* lab;
  long long lab_nrec;
  int lab_set;
  bool global = false;    // win is the device table in global memory: read-only loads, 64-bit index
  // stochastic forcing (samsim_b200_set_stochastic_forcing): this column's perturbed record values of the launch's
  // window, cw[((rec - win_first)*4 + kind)*cw_ld], written by samsim_noise_kernel; nullptr = read the table
  const double* cw = nullptr;
  long long cw_ld;
};

__device__ __forceinline__ double forcing_rec(const Forcing& f, int kind, int rec /*1-based*/) {
#ifdef __CUDA_ARCH__
  if (f.cw) return __ldg(f.cw + ((long long)(rec - f.win_first) * 4 + kind) * f.cw_ld);
  // (site*4 + kind)*nrec passes 2^31 at about 183,000 sites of a year of 3-hourly records
  const double base = f.global ? __ldg(f.win + (((long long)f.site * 4 + kind) * f.win_len + (rec - f.win_first)))
                               : f.win[(f.site * 4 + kind) * f.win_len + (rec - f.win_first)];
#else
  if (f.cw) return f.cw[((long long)(rec - f.win_first) * 4 + kind) * f.cw_ld];
  const double base = f.win[((long long)f.site * 4 + kind) * f.win_len + (rec - f.win_first)];
#endif
  return base * f.scale[kind] + f.offset[kind];
}
// time_input(k) = (REAL(k)-1._wp)*3600._wp*3._wp, mo_functions.f90:323-325
__device__ __forceinline__ double time_input(int k) { return ((double)(float)k - 1.0) * 3600.0 * 3.0; }
__device__ __forceinline__ double lab_rec(const Forcing& f, int kind, long long rec /*1-based*/) {
  return f.lab[((long long)(f.lab_set * 4 + kind)) * f.lab_nrec + (rec - 1)];
}

// S0 vital signs, mo_grotz.f90:192-223 (diagnostics; psi_* are the previous step's)
__device__ __noinline__ void vital_signs(Col& c) {
  const View v = c;
  const int Na = c.N_active;
  double sumH = 0.0, summ = 0.0, sumS = 0.0;
  SAMSIM_LOOP
  for (int k = 1; k <= Na; k++) { sumH = sumH + v.H_abs()[k]; summ = summ + v.m()[k]; sumS = sumS + v.S_abs()[k]; }
  SCV(c, SC_ENERGY_STORED) = SCV(c, SC_H_ABS_SNOW) + sumH - SCV(c, SC_T_BOTTOM) * summ * c_l;
  double fw = summ / rho_l;
  fw = fw * (1.0 - sumS / summ / ref_salinity);
  fw = fw + SCV(c, SC_M_SNOW) / rho_l;
  SCV(c, SC_FRESHWATER) = fw;
  double tr = 0.0;
  SAMSIM_LOOP
  for (int jj = 1; jj <= Na - 1; jj++) tr = tr + v.thick()[jj] / (v.psi_l()[jj] * k_l + v.psi_s()[jj] * k_s);
  const double thNa = v.thick()[Na], psNa = v.psi_s()[Na];
  tr = tr + thNa * psNa / psi_s_min * (psi_s_min * k_s + 1.0 - psi_s_min * k_l);
  if (SCV(c, SC_THICK_SNOW) > CFG.thick_min / 110.0) tr = tr + SCV(c, SC_THICK_SNOW) / k_snow_of(SCV(c, SC_M_SNOW), SCV(c, SC_THICK_SNOW));
  SCV(c, SC_TOTAL_RESIST) = tr;
  double th = (Na > 1) ? sum_fwd(v.thick(), 1, Na - 1) : 0.0;
  SCV(c, SC_THICKNESS) = th + thNa * psNa / psi_s_min;
  if (Na > 1) {
    double b = sum_fwd(v.S_abs(), 1, Na - 1) + v.S_abs()[Na] * psNa / psi_s_min;
    b = b / (sum_fwd(v.m(), 1, Na - 1) + v.m()[Na] * psNa / psi_s_min);
    SCV(c, SC_BULK_SALIN) = b;
  } else {
    SCV(c, SC_BULK_SALIN) = v.S_abs()[1] / v.m()[1];
  }
}

// Surface part of sub_heat_fluxes, mo_heat_fluxes.f90:77-258: the flux into layer 1 (returned), T_top, albedo, the snow
// flux and fl_rad(N_active).  Shared by the sub-step-by-sub-step path (heat_fluxes) and the merged forward pass
// (forward_pass), so both evaluate the same expressions.  Layer-1 / bottom-layer inputs are passed by value.
struct SurfIn {
  double ps1, pl1, pg1, th1, T1;   // psi_s(1), psi_l(1), psi_g(1), thick(1), T(1)
  double S1, m1, SNa, mNa;         // S_abs / m of layer 1 and layer N_active as they are when sub_heat_fluxes runs
  double flQ1_prev;                // fl_Q(1) of the previous step (kept when no boundflux branch assigns it)
};
__device__ __noinline__ double heat_surface(Col& c, const SurfIn& in, double& fl_rad_Na) {
  const View v = c;
  const int Na = c.N_active;
  const double thick_min = CFG.thick_min;
  const double ps1 = in.ps1, pl1 = in.pl1, pg1 = in.pg1, th1 = in.th1, T1 = in.T1;
  double& thick_snow = SCV(c, SC_THICK_SNOW);
  double& T_top = SCV(c, SC_T_TOP);
  double& fl_q_snow = SCV(c, SC_FL_Q_SNOW);
  double flQ1 = in.flQ1_prev;
  fl_rad_Na = 0.0;  // fl_rad(N_active): 0 unless boundflux 2 recomputes it (fl_rad = 0 from init, mo_init.f90:1988)

  if (CFG.boundflux_flag == 1) {  // :77-86
    flQ1 = fl_Q_0_top(ps1, pl1, pg1, th1, T1, T_top);
    if (fabs(flQ1) > CFG.max_flux_plate) flQ1 = flQ1 / fabs(flQ1) * CFG.max_flux_plate;
  }

  if (CFG.boundflux_flag == 2) {  // :90-195
    double& albedo = SCV(c, SC_ALBEDO);
    double& fl_sw = SCV(c, SC_FL_SW);
    double& fl_rest = SCV(c, SC_FL_REST);
    albedo = albedo_of(thick_snow, SCV(c, SC_T_SNOW), pl1, thick_min, CFG.albedo_flag);
    if (CFG.atmoflux_flag == 1) {
      EVT(c, EV_NOTZFLUX);
      notzflux(c.time + 86400.0 * 180.0, fl_sw, fl_rest);
    } else if (CFG.atmoflux_flag == 2) {  // :97-111
      double fl_lw;
      if (c.time == c.ftime1) {
        fl_sw = c.fsw1;
        fl_lw = c.flw1;
      } else {
        const double temp = (c.time - c.ftime0) / (c.ftime1 - c.ftime0);
        fl_sw = (1.0 - temp) * c.fsw0 + temp * c.fsw1;
        fl_lw = (1.0 - temp) * c.flw0 + temp * c.flw1;
      }
      SCV(c, SC_FL_LW) = fl_lw;
      fl_rest = fl_lw + 0.0 + 0.0;  // fl_sen = fl_lat = 0
    }
    double T_old, emi, pen;
    if (thick_snow < thick_min) { T_old = T1; emi = emissivity_ice; pen = penetr; }
    else { T_old = SCV(c, SC_T_SNOW); emi = emissivity_snow; pen = 0.0; }
    T_old = T_old + zeroK;
    double temp1 = (1.0 - albedo) * (1.0 - pen) * fl_sw + fl_rest;  // :135-139
    temp1 = temp1 + emi * 3.0 * sigma * P4(T_old);
    temp1 = temp1 / (emi * 4.0 * sigma * P3(T_old));
    temp1 = temp1 - zeroK;
    T_old = temp1 + zeroK;  // :141-146
    temp1 = (1.0 - albedo) * (1.0 - pen) * fl_sw + fl_rest;
    temp1 = temp1 + emi * 3.0 * sigma * P4(T_old);
    temp1 = temp1 / (emi * 4.0 * sigma * P3(T_old));
    temp1 = temp1 - zeroK;
    T_top = temp1;

    // :151-155 Beer law.  Only fl_rad(N_active) is ever read (:283-284), but the running product
    // must see every layer in order.  exp() of a repeated thickness is reused (same bits).
    {
      double temp2 = pen * (1.0 - albedo) * fl_sw;
      double last_th = -1.0, last_e = 0.0;
      // no penetrating short wave (polar night, or snow: pen = 0): 0 - 0*exp(..) = 0 and the product stays 0
      const int kend = (temp2 == 0.0) ? 0 : Na;
      SAMSIM_LOOP
      for (int k = 1; k <= kend; k++) {
        if (k + SAMSIM_PF <= Na) v.thick().prefetch(k + SAMSIM_PF);
        const double thk = v.thick()[k];
        if (thk != last_th) { last_e = det_exp(-extinc * thk); last_th = thk; }
        if (k == Na) fl_rad_Na = temp2 - temp2 * last_e;
        temp2 = temp2 * last_e;
      }
    }

    double& T_freeze = SCV(c, SC_T_FREEZE);
    if (thick_snow >= thick_min / 100.0) T_freeze = 0.0;  // :158-162
    else T_freeze = T_freeze_of(in.S1 / in.m1, CFG.salt_flag);

    if (T_top > T_freeze && Na > 1) {  // :167-180
      EVT(c, EV_HEAT_MELT);
      temp1 = emi * sigma * P4(T_freeze + zeroK) - (1.0 - albedo) * (1.0 - pen) * fl_sw - fl_rest;
      if (thick_snow >= thick_min) {
        fl_q_snow = temp1;
        flQ1 = fl_Q_snow_ice(SCV(c, SC_M_SNOW), thick_snow, SCV(c, SC_T_SNOW), ps1, pl1, th1, T1);
      } else if (thick_snow >= thick_min / 100.0) {
        fl_q_snow = temp1;
        flQ1 = 0.0;
      } else {
        flQ1 = temp1;
      }
      T_top = T_freeze;
    } else {  // :185-193
      if (thick_snow >= thick_min) {
        flQ1 = fl_Q_snow_ice(SCV(c, SC_M_SNOW), thick_snow, SCV(c, SC_T_SNOW), ps1, pl1, th1, T1);
        fl_q_snow = fl_Q_0_snow(SCV(c, SC_M_SNOW), thick_snow, SCV(c, SC_T_SNOW), T_top);
      } else if (thick_snow > thick_min / 100.0 && thick_snow < thick_min) {
        flQ1 = 0.0;
        fl_q_snow = fl_Q_0_snow_thin(SCV(c, SC_M_SNOW), thick_snow, SCV(c, SC_T_SNOW), ps1, pl1, pg1, th1, T_top);
      } else {
        flQ1 = fl_Q_0_top(ps1, pl1, pg1, th1, T1, T_top);
      }
    }
  }

  if (CFG.boundflux_flag == 3) {  // :202-258
    const double T2m = SCV(c, SC_T2M);
    double& T_freeze = SCV(c, SC_T_FREEZE);
    if (CFG.lab_snow_flag == 0 || thick_snow <= thick_min / 100.0) {
      T_freeze = f_min(T_freeze_of(in.SNa / in.mNa, CFG.salt_flag), 0.0);
      T_top = T1;
      flQ1 = CFG.alpha_flux_instable * (T_top - T2m);
      if (flQ1 < 0.0) {
        T_top = f_max(T_freeze, T1);
        flQ1 = CFG.alpha_flux_stable * (T_top - T2m);
      }
      if (thick_snow == 0.0 && CFG.lab_snow_flag == 1 && c.styropor_flag == 1) {  // sub_fl_Q_styropor, mo_thermo_functions.f90:276
        EVT(c, EV_STYROPOR);
        flQ1 = flQ1 * CFG.k_styropor;
      }
    } else if (CFG.lab_snow_flag == 1) {
      T_freeze = T_freeze_of(SCV(c, SC_S_ABS_SNOW) / SCV(c, SC_M_SNOW), CFG.salt_flag);
      T_top = SCV(c, SC_T_SNOW);
      double temp1 = CFG.alpha_flux_instable * (T_top - T2m);
      if (temp1 >= 0.0) {
        if (thick_snow >= thick_min) {
          fl_q_snow = temp1;
          flQ1 = fl_Q_snow_ice(SCV(c, SC_M_SNOW), thick_snow, SCV(c, SC_T_SNOW), ps1, pl1, th1, T1);
        } else if (thick_snow >= thick_min / 100.0) {
          fl_q_snow = fl_Q_0_snow_thin(SCV(c, SC_M_SNOW), thick_snow, SCV(c, SC_T_SNOW), ps1, pl1, pg1, th1, (T2m + T_top) / 2.0);
          flQ1 = 0.0;
        }
      } else {
        temp1 = CFG.alpha_flux_stable * (T_top - T2m);
        if (thick_snow >= thick_min) {
          fl_q_snow = temp1;
          flQ1 = fl_Q_snow_ice(SCV(c, SC_M_SNOW), thick_snow, SCV(c, SC_T_SNOW), ps1, pl1, th1, T1);
        } else if (thick_snow >= thick_min / 100.0) {
          fl_q_snow = temp1;
          flQ1 = 0.0;
        }
      }
    }
  }

  return flQ1;
}

// sub_heat_fluxes, mo_heat_fluxes.f90:69-312
__device__ __noinline__ void heat_fluxes(Col& c) {
  const View v = c;
  const int Na = c.N_active;
  const double dt = CFG.dt, thick_min = CFG.thick_min;
  const double ps1 = v.psi_s()[1], pl1 = v.psi_l()[1], pg1 = v.psi_g()[1], th1 = v.thick()[1];
  double T1 = v.T()[1];
  const double thick_snow = SCV(c, SC_THICK_SNOW);
  double fl_rad_Na;
  const SurfIn in = {ps1, pl1, pg1, th1, T1, v.S_abs()[1], v.m()[1], v.S_abs()[Na], v.m()[Na], v.fl_Q()[1]};
  const double flQ1 = heat_surface(c, in, fl_rad_Na);
  const double fl_q_snow = SCV(c, SC_FL_Q_SNOW);

  const double fl_q_bottom = SCV(c, SC_FL_Q_BOTTOM);
  v.fl_Q()[1] = flQ1;
  v.fl_Q()[Na + 1] = fl_q_bottom;  // :262 (every step: it is the entry that stays behind when N_active shrinks)

  // :269-285 in one forward pass: energy sums (forward order), inter-layer fluxes, explicit update.
  double temp1 = 0.0, temp2 = 0.0;
  {
    double fq_k = flQ1;
    // sub_fl_Q (mo_thermo_functions.f90:201-224): R = thick_1/(2 k_1) + thick_2/(2 k_2).  The half resistance of a
    // layer is the same expression whether the layer is the upper or the lower one of a pair, so it is evaluated
    // once per layer and carried (one division per layer instead of two, same bits).
    double hr_k = th1 / (2.0 * (ps1 * k_s + pl1 * k_l + pg1 * 0.0)), T_k = T1;
    const double rad = fl_rad_Na * dt;
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) {
      if (k + 1 + SAMSIM_PF <= Na) {
        const int kp = k + 1 + SAMSIM_PF;
        v.psi_s().prefetch(kp); v.psi_l().prefetch(kp); v.thick().prefetch(kp); v.T().prefetch(kp);
        v.H_abs().prefetch(kp);
      }
      double fq_kp1;
      double hr_n = 0.0, T_n = 0.0;
      if (k < Na) {
        // psi_g enters k = psi_s*k_s + psi_l*k_l + psi_g*0._wp only as +-0 (psi_g is a finite volume fraction, k > 0)
        const double ps_n = v.psi_s()[k + 1], pl_n = v.psi_l()[k + 1], th_n = v.thick()[k + 1];
        T_n = v.T()[k + 1];
        hr_n = th_n / (2.0 * (ps_n * k_s + pl_n * k_l + 0.0 * 0.0));
        const double R = hr_k + hr_n;
        fq_kp1 = (T_n - T_k) / R;  // :272-274
        if (c.want_state) v.fl_Q()[k + 1] = fq_kp1;  // fl_Q(2:N_active) is never read back by the loop body; N_active moves by
                                                     // at most 1 per step, so a stale interior entry is always overwritten by a later :262
      } else {
        fq_kp1 = fl_q_bottom;
      }
      double H = v.H_abs()[k];
      temp1 = temp1 + H;                 // :269 sum(H_abs) before the update
      H = H + (fq_kp1 - fq_k) * dt;      // :277-279
      H = H + rad;                       // :282-285 (sic: fl_rad(N_active) for every layer)
      v.H_abs()[k] = H;
      temp2 = temp2 + H;                 // :305 sum(H_abs) after the update (layer 1 re-added below if coupling changes it)
      fq_k = fq_kp1;
      hr_k = hr_n; T_k = T_n;
    }
    temp1 = temp1 + SCV(c, SC_H_ABS_SNOW);
    SAMSIM_LOOP
    for (int k = 1; k <= Na; k++) temp1 = temp1 + rad;  // :284 temp1 = temp1 + fl_rad(N_active)*dt, N_active times
  }

  bool layer1_changed = false;
  if (thick_snow >= thick_min / 100.0 && thick_snow < thick_min) {  // :291-295
    EVT(c, EV_HEAT_THIN_SNOW);
    SCV(c, SC_H_ABS_SNOW) = SCV(c, SC_H_ABS_SNOW) - fl_q_snow * dt;
    double H1 = v.H_abs()[1], phi1 = v.phi()[1];
    snow_coupling(c, H1, phi1, T1, v.m()[1], v.S_bu()[1]);
    v.H_abs()[1] = H1; v.phi()[1] = phi1; v.T()[1] = T1;
    layer1_changed = true;
    temp1 = temp1 + fl_q_bottom * dt - fl_q_snow * dt;
  } else if (thick_snow >= thick_min) {  // :296-299
    SCV(c, SC_H_ABS_SNOW) = SCV(c, SC_H_ABS_SNOW) + (flQ1 - fl_q_snow) * dt;
    temp1 = temp1 + fl_q_bottom * dt - fl_q_snow * dt;
  } else {
    temp1 = temp1 + fl_q_bottom * dt - flQ1 * dt;  // :302
  }
  if (layer1_changed) temp2 = sum_fwd(v.H_abs(), 1, Na);  // forward order requires a fresh pass when H_abs(1) moved
  temp2 = temp2 + SCV(c, SC_H_ABS_SNOW);
  if (fabs((temp1 - temp2) / dt) > 0.00001) c.status = 431;  // :307-310
}

// One loop iteration.  `last_of_launch` makes the S0 diagnostics observable through get_scalar
// (they are otherwise only consumed by S8); `snap` receives the S8 record.
// Phase synchronisation: with SAMSIM_SYNC=1 every warp of the block passes the same barrier between groups of
// sub-steps, so all warps of the block execute the same few KB of code at the same time.  The step kernel is
// ~300 KB of SASS and instruction fetch (stall_no_instruction), not the FP64 pipe, limits it otherwise.  The
// barriers sit at block-uniform points: failed / padding columns skip the phase bodies but not the barriers.
#ifndef SAMSIM_SYNC
#define SAMSIM_SYNC 1
#endif
// S_bu is rewritten by S4 / S7 before anything reads it; only its value after the last step of a launch is observable
#ifndef SAMSIM_ALWAYS_STORE_S_BU
#define SAMSIM_ALWAYS_STORE_S_BU false
#endif
#if SAMSIM_SYNC
#define SAMSIM_PHASE_SYNC() __syncthreads()
#else
#define SAMSIM_PHASE_SYNC() ((void)0)
#endif
#if SAMSIM_SYNC >= 2
#error "SAMSIM_SYNC=2 (a barrier per layer of the Newton sweeps) was removed: it measured slower and its fused / unfused \
choice per thread made the barrier divergent (ADVICE round 1)"
#endif

struct SnapOut {
  double* scalars;  // [SNAPSC_COUNT][ncol_pad] or nullptr
  double* arrays;   // [SNAPARR_COUNT][Nlayer+2][ncol_pad] or nullptr
  size_t ncol_pad;
  int col;
};

__device__ __noinline__ void write_snapshot(const Col& c, const SnapOut& s) {
  const View v = c;
  if (s.scalars) {
    const int ids[19] = {SC_FREEBOARD, SC_THICK_SNOW, SC_T_SNOW, SC_PSI_L_SNOW, SC_PSI_S_SNOW, SC_ENERGY_STORED,
                         SC_FRESHWATER, SC_TOTAL_RESIST, SC_THICKNESS, SC_BULK_SALIN, SC_GRAV_DRAIN, SC_GRAV_SALT,
                         SC_GRAV_TEMP, SC_T2M, SC_T_TOP, SC_MTO1, SC_MTO2, SC_MTO3, -1};
    SAMSIM_LOOP
    for (int q = 0; q < 18; q++) s.scalars[(size_t)q * s.ncol_pad + s.col] = c.sc[ids[q]];
    s.scalars[(size_t)18 * s.ncol_pad + s.col] = c.time;
    s.scalars[(size_t)19 * s.ncol_pad + s.col] = (double)c.N_active;
  }
  if (s.arrays) {
    const int N = CFG.Nlayer;
    const size_t LS = (size_t)(N + 2);
    const int src[10] = {AR_T, AR_PSI_S, AR_THICK, AR_S_BU, AR_RAY, AR_PSI_L, AR_PERM, AR_FLUSH_V, AR_FLUSH_H, AR_PSI_G};
    SAMSIM_LOOP
    for (int a = 0; a < 10; a++) {
      double* dst = s.arrays + ((size_t)a * LS) * s.ncol_pad + s.col;
      const Lay from = v.A(src[a]);
      const int n = (a == 4) ? N - 1 : N;
      SAMSIM_LOOP
      for (int k = 1; k <= n; k++) dst[(size_t)k * s.ncol_pad] = from[k];
    }
    for (int q = 0; q < CFG.n_bgc; q++) {  // output_bgc, mo_output.f90:165-186
      double* bu = s.arrays + ((size_t)(10 + 2 * q) * LS) * s.ncol_pad + s.col;
      double* br = s.arrays + ((size_t)(11 + 2 * q) * LS) * s.ncol_pad + s.col;
      const Lay x = v.bgc(q);
      const double bottom = c.sc[SC_BGC_BOTTOM1 + q];
      SAMSIM_LOOP
      for (int k = 1; k <= N; k++) {
        double vbu = bottom, vbr = bottom;
        if (k <= c.N_active) {
          const double mk = v.m()[k];
          if (mk != 0.0) {
            vbu = x[k] / mk;
            const double pl = v.psi_l()[k], th = v.thick()[k];
            vbr = (pl != 0.0 && th != 0.0) ? x[k] / pl / th / rho_l : 0.0;
          } else {
            vbu = 0.0; vbr = 0.0;
          }
        }
        bu[(size_t)k * s.ncol_pad] = vbu;
        br[(size_t)k * s.ncol_pad] = vbr;
      }
    }
  }
}

// S4 + S5 + S7 in ONE forward pass.  Precondition: layers 2..N_active carry the T and phi of a getT sweep over their
// current m, S_abs, H_abs -- the S18 sweep of the previous step when nothing touched them since (c.thermo_valid),
// otherwise the same sweep run just before (column_step, phase 1) -- so S4 has no backward dependency left.
// Per layer: S_br and the volume fractions (S4, :298-307), expulsion_flux (mo_mass.f90:112-136), mass_transfer
// (mo_mass.f90:53-96, skipped at i == 1) and S_bu = S_abs/m (S7, :333-335), with fl_m and V_ex carried in registers
// instead of being written and re-read.  Same operations in the same order as the three separate sweeps:
//   * expulsion_flux finishes before mass_transfer starts in the reference, but mass_transfer reads neither m
//     nor psi_g, and expulsion_flux reads neither H_abs nor S_abs;
//   * mass_transfer(k) evaluates S_br from the S4 values T, S_bu of layers k-1 and k: S_br(k) is computed once and
//     carried; S7 overwrites S_bu(k) after mass_transfer(k) used the S4 value.
__device__ __noinline__ void fused_thermo_expulsion(Col& c) {
  const View v = c;
  const int Na = c.N_active;
  const bool transfer = (c.i != 1);
  {  // layer 1 is always recomputed; its first guess is T(2) of the (valid) sweep, T_bottom when it is the only layer
    const double m1 = v.m()[1];
    const double sbu1 = v.S_abs()[1] / m1, H = v.H_abs()[1] / m1;
    double phi1 = v.phi()[1], T1;
    const double T_test = (Na >= 2) ? v.T()[2] : SCV(c, SC_T_BOTTOM);
    getT(H, sbu1, T_test, T1, phi1, c.status, c.ev1);
    v.T()[1] = T1; v.phi()[1] = phi1;
  }
  // expulsion_flux only produces fl_m <= 0 (see expel_layer below): of mass_transfer's four branches only
  // `fl_m(k+1) < 0` and `fl_m(k) < 0` can be taken, the layer below is never read, and the pass needs no look-ahead.
  // Carried from layer k-1: T, S_br (the S4 value mass_transfer evaluates again from the same T and S_bu,
  // mo_mass.f90:91), the S_abs the transfer left there, fl_m(k).
  double T_km1 = 0.0, sbr_km1 = 0.0, Sabs_km1 = 0.0, f0 = 0.0;
  // func_freeboard memo: forward totals and the exact suffix sums for the waterline layer of the previous step
  double fbA = 0.0, fbG = 0.0, fbAs = 0.0, fbGs = 0.0;
  const int ks = (c.fb.k_last >= 1 && c.fb.k_last < Na) ? c.fb.k_last : 0;
  double min_ps = 1e300;
  SAMSIM_LOOP
  for (int k = 1; k <= Na; k++) {
    if (k + SAMSIM_PF <= Na) {
      v.T().prefetch(k + SAMSIM_PF); v.phi().prefetch(k + SAMSIM_PF);
      v.m().prefetch(k + SAMSIM_PF); v.thick().prefetch(k + SAMSIM_PF); v.S_abs().prefetch(k + SAMSIM_PF);
      v.H_abs().prefetch(k + SAMSIM_PF);
    }
    const double thk = v.thick()[k], m_k = v.m()[k], T_k = v.T()[k];
    double S = v.S_abs()[k];
    // S4: S_bu = S_abs/m (:299; the S_bu array is not kept current by the S18 sweep), brine salinity, volume fractions
    const double sbr_k = S_br_of(T_k, S / m_k);
    v.S_br()[k] = sbr_k;
    double ps, pl, pg, vex;
    expulsion(v.phi()[k], thk, m_k, ps, pl, pg, vex);
    // expulsion_flux, mo_mass.f90:121-134
    double f1;
    if (k == 1) {
      f1 = -vex * rho_l;
    } else if (pg < SAMSIM_F32(0.001)) {
      f1 = -vex * rho_l + f0;
    } else {
      f1 = -f_max((vex - pg * thk) * rho_l, 0.0);
      pg = f_max((pg * thk - vex) / thk, 0.0);
    }
    v.psi_s()[k] = ps; v.psi_l()[k] = pl; v.psi_g()[k] = pg;
    fbA = fbA + ps * thk;
    fbG = fbG + pg * thk;
    if (ks && k > ks) { fbAs = fbAs + ps * thk; fbGs = fbGs + pg * thk; }
    min_ps = f_min(min_ps, ps);
    const double m_new = m_k + f1 - f0;
    v.m()[k] = m_new;
    // mass_transfer layer k (mo_mass.f90:82-84, :89-92), then S7
    if (transfer) {
      double H = v.H_abs()[k];
      if (f1 < 0.) {
        H = H + f1 * T_k * c_l;
        S = S + f_max(f1 * sbr_k, -S);
      }
      if (f0 < 0) {
        H = H - f0 * T_km1 * c_l;
        S = S - f_max(f0 * sbr_km1, -Sabs_km1);
      }
      v.H_abs()[k] = H;
      v.S_abs()[k] = S;
    }
    v.S_bu()[k] = S / m_new;
    if (CFG.n_bgc) {  // mo_grotz.f90:316-320: fl_brine_bgc(k,k+1) = -fl_m(k+1); the other cells start the step empty
      v.A(AR_FB_D)[k] = transfer ? -f1 : 0.0;
      v.A(AR_FB_U)[k] = 0.0; v.A(AR_FB_A)[k] = 0.0; v.A(AR_FB_O)[k] = 0.0;
    }
    T_km1 = T_k; sbr_km1 = sbr_k; Sabs_km1 = S;
    f0 = f1;
  }
  c.fb.tot_valid = true; c.fb.t1 = v.thick()[1]; c.fb.A = fbA; c.fb.G = fbG;
  c.fb.suf_valid = (ks != 0); c.fb.ks = ks; c.fb.As = fbAs; c.fb.Gs = fbGs;
  c.fb.res_valid = false;
  c.min_psi_s = min_ps;
}

// S15 testcase hooks, mo_grotz.f90:503-563
__device__ __forceinline__ void testcase_hooks(Col& c, const Forcing& f) {
  const View v = c;
  const double dt = CFG.dt;
  const int N = CFG.Nlayer;
  if (CFG.testcase == 1) {  // sub_test1, mo_testcase_specifics.f90:42-89
    const double j = rint(c.time / 43200.0);
    if (j >= 1.0 && j <= 20.0 && fabs(c.time - 12.0 * j * 3600.0) < SAMSIM_F32(0.01))
      SCV(c, SC_T_TOP) = (((int)j) & 1) ? SCV(c, SC_TTOP_COLD) : SCV(c, SC_TTOP_WARM);
  } else if (CFG.testcase >= 101 && CFG.testcase <= 105) {  // :521-530
    const long long idx = (long long)floor(1 + c.time / dt);
    const double Sb = v.S_bu()[c.N_active + 1];
    SCV(c, SC_T2M) = lab_rec(f, 0, idx);
    SCV(c, SC_SOLID_PRECIP) = lab_rec(f, 1, idx);
    SCV(c, SC_FL_Q_BOTTOM) = lab_rec(f, 2, idx);
    SCV(c, SC_T_BOTTOM) = -SAMSIM_F32(0.0575) * Sb + SAMSIM_F32(1.710523e-3) * det_pow(Sb, 3.0 / 2.0) -
                          SAMSIM_F32(2.154996e-4) * P2(Sb) - SAMSIM_F32(7.53e-4) * sum_fwd(v.thick(), 1, c.N_active - 1);
    c.styropor_flag = (int)lab_rec(f, 3, idx);
  } else if (CFG.testcase == 4 || CFG.testcase == 7) {  // sub_test4, mo_testcase_specifics.f90:197-202
    const double amp = SCV(c, SC_OFLUX_AMP);
    SCV(c, SC_FL_Q_BOTTOM) = -amp * det_sin(c.time * (2.0 * pi_sp) / (86400.0 * 365.0)) + amp;
  } else if (CFG.testcase == 2) {  // sub_test2, mo_testcase_specifics.f90:92-101
    if (c.time > 86400.0 * 25.0) SCV(c, SC_T2M) = 15.0;
    else if (c.time > 86400.0 * 15.0) SCV(c, SC_T2M) = 1.0;
  } else if (CFG.testcase == 9) {  // sub_test9, :105-116
    if (c.time < (19.75 * 3600.0)) SCV(c, SC_T2M) = 0.0;
    else if (c.time < (86400.0 * 3.0 + 2.25 * 3600.0)) SCV(c, SC_T2M) = -15.0;
    else SCV(c, SC_T2M) = 1.0;
  } else if (CFG.testcase == 34) {  // sub_test34, :146-161
    if (c.time < 2.0 * 3600.0) SCV(c, SC_T2M) = 0.0;
    else if (c.time < (86400.0 * 5.0)) SCV(c, SC_T2M) = -15.0;
    else if (c.time < (86400.0 * 7.0)) SCV(c, SC_T2M) = -5.0;
    else SCV(c, SC_T2M) = 1.0;
  } else if (CFG.testcase == 99) {  // mo_grotz.f90:547-563: from day 3 on the snow cover is reset every step
    if (c.time < 86400.0 * 3.0) {
      SCV(c, SC_T2M) = -40.0;
    } else {
      SCV(c, SC_T2M) = (c.time > 86400.0 * 5.0) ? 5.0 : -5.0;
      SCV(c, SC_THICK_SNOW) = 0.2;
      SCV(c, SC_T_SNOW) = -5.0;
      SCV(c, SC_M_SNOW) = 30.0;
      SCV(c, SC_H_ABS_SNOW) = -SCV(c, SC_M_SNOW) * latent_heat;
    }
  } else if (CFG.testcase == 3) {  // sub_test3, :170-185
    SCV(c, SC_LIQUID_PRECIP) = 0.0;
    SCV(c, SC_SOLID_PRECIP) = 0.15 / 86400.0 / 356.0;
  } else if (CFG.testcase == 6) {  // sub_test6, :218-243
    const double t = c.time;
    if (t > 1714.0 * 60.0) SCV(c, SC_T2M) = -19.0;
    else if (t > 1676.0 * 60.0) SCV(c, SC_T2M) = -5.0;
    else if (t > 1525.0 * 60.0) SCV(c, SC_T2M) = -18.0;
    else if (t > 1483.0 * 60.0) SCV(c, SC_T2M) = -5.0;
    else if (t > 1385.0 * 60.0) SCV(c, SC_T2M) = -18.0;
    else if (t > 1349.0 * 60.0) SCV(c, SC_T2M) = -5.0;
    else if (t > 1160.0 * 60.0) SCV(c, SC_T2M) = -18.0;
    else if (t > 1100.0 * 60.0) SCV(c, SC_T2M) = -5.0;
  } else if (CFG.testcase == 111) {  // mo_grotz.f90:505-506: harp temperatures, one record per time step
    SCV(c, SC_T_TOP) = lab_rec(f, 0, (long long)floor(1 + c.time / dt));
  } else if (CFG.testcase == 8) {  // mo_grotz.f90:539-544: field temperatures, one record per minute, until day 5.5
    if (c.time < (double)(3600.f * 12.f * 11.f)) SCV(c, SC_T_TOP) = lab_rec(f, 0, (long long)floor(1 + c.time / 60));
    else SCV(c, SC_T_TOP) = -15.0;
  } else if (CFG.testcase == 5 && c.i == 2) {  // mo_grotz.f90:541-542
    SAMSIM_LOOP
    for (int k = 1; k <= N; k++) v.S_abs()[k] = 5.0 * v.m()[k];
  }

}

// ==========================================================================================================
// The two-pass step.  In the steady regime (no flooding, no flushing, no layer event, a proper snow layer or none)
// a model step touches the per-layer arrays in exactly two sweeps instead of five:
//
//   forward_pass   k = 1..N_active   S4 (layer 1 getT; layers >= 2 reuse the S18 result), S5 expulsion_flux +
//                                    mass_transfer, S7, S9, S12, S13 fl_grav_drain incl. its mass_transfer, S17
//                                    sub_heat_fluxes -- merged with a lag of one layer (layer k-1 is finished while
//                                    layer k is expelled and drained)
//   backward_pass  k = N_active..1   S18 getT sweep, plus the layer-local half of the NEXT step's fl_grav_drain
//                                    (permeability, thick/perm, suffix estimates of the Rayleigh numbers)
//
// Per layer and step the forward pass reads m, S_abs, H_abs, thick, T, phi, ray (7) and writes m, S_abs, H_abs, psi_s,
// psi_l, psi_g (6); the backward pass reads m, S_abs, H_abs, thick (4) and writes T, phi, ray, thick/perm (4): 21
// array passes instead of 37.  S_br, V_ex, fl_m, S_bu, fl_Q(2:) never leave the registers.  Every value is computed by
// the same expression, in the same order, as in the sub-step-by-sub-step path below (and in the reference); the
// bitwise parity tests run both.  column_step takes this path only when fast_path_ok() holds; everything else --
// output steps, the last step of a launch (whose ray / S_bu / fl_Q arrays are observable), thin snow, possible
// flooding, tracers, tank / lab cases -- goes through the general path.
// ==========================================================================================================

// S18, mo_grotz.f90:592-598 (psi_* are NOT refreshed).  `prepare`: also evaluate, for layers 2..N_active, what the
// next step's S4 and fl_grav_drain (mo_grav_drain.f90:104-136) will compute from T, phi, m, thick, S_abs of the layer
// alone: Expulsion -> psi_l -> perm, thick/perm (stored in w1), and the suffix estimates of ray (stored in ray, see
// grav_drain for the estimate / candidate scheme).  Only done when ray is not observable before it is recomputed.
// PREP is a template parameter: the general-path kernel is instantiated without the preparation code (and without
// forward_pass): compiled into one kernel, the unused two-pass code cost the general path 10 % (instruction cache).
template <bool PREP>
__device__ __noinline__ void backward_pass(Col& c, bool prepare_now, bool store_S_bu) {
  const bool prepare = PREP && prepare_now;
  const View v = c;
  const int Na = c.N_active;
  Lay q = v.w1();
  double T_test = SCV(c, SC_T_BOTTOM);
  double min_S2 = 1e300;
  double mn = 0.0, sq = 0.0, st = 0.0, bottom_h = 0.0, S_br_Na = 0.0, perm_Na = 0.0, qb_est = 0.0, A2 = 0.0;
  SAMSIM_LOOP
  for (int k = Na; k >= 1; k--) {
    if (k - SAMSIM_PF >= 1) {
      v.m().prefetch(k - SAMSIM_PF); v.S_abs().prefetch(k - SAMSIM_PF); v.H_abs().prefetch(k - SAMSIM_PF);
      if (prepare) v.thick().prefetch(k - SAMSIM_PF);
    }
    const double mk = v.m()[k];
    const double Sk = v.S_abs()[k];
    if (k >= 2) min_S2 = f_min(min_S2, Sk);
    const double sbu = Sk / mk;
    const double H = v.H_abs()[k] / mk;
    double T, phi;
    if (!getT_body(H, sbu, T_test, T, phi, c.status, c.ev1)) phi = v.phi()[k];  // inlined: no call, no spills in the hot sweep
    T_test = T;
    v.T()[k] = T; v.phi()[k] = phi;
    if (store_S_bu) v.S_bu()[k] = sbu;
    if (prepare && k >= 2) {
      const double thk = v.thick()[k];
      double ps, pl, pg, vex;
      expulsion(phi, thk, mk, ps, pl, pg, vex);                       // S4 of the next step, :298-307
      A2 = A2 + ps * thk;
      const double pk = 1e-17 * det_pow(1000.0 * fabs(pl), 3.10);     // mo_grav_drain.f90:104-106
      const double sbr = S_br_of(T, sbu);
      if (k == Na) {
        perm_Na = pk; bottom_h = thk * ps / psi_s_min; qb_est = bottom_h / pk; S_br_Na = sbr;
      } else {
        const double qk = thk / pk;
        q[k] = qk;
        mn = (k == Na - 1) ? pk : f_min(mn, pk);
        const double st_below = st;
        sq = sq + qk;
        st = st + thk;
        const double hp = (mn < 1e-14) ? 0.0 : (st + bottom_h) / (sq + qb_est);
        double est = grav * rho_l * bbeta * (sbr - S_br_Na) * (st_below + bottom_h) * hp;
        est = est / (kappa_l * mu);
        v.ray()[k] = (mn < 1e-14) ? 0.0 : f_max(est, 0.0);
      }
    }
  }
  c.min_S_abs_2 = min_S2;
  c.thermo_valid = true;  // invalidated by anything that touches layers >= 2
  c.pre.valid = prepare;
  c.pre.mn2 = mn; c.pre.sq2 = sq; c.pre.st2 = st; c.pre.bottom_h = bottom_h; c.pre.S_br_Na = S_br_Na; c.pre.perm_Na = perm_Na;
  c.pre.A2 = A2;
}

// The two-pass step is selected per handle at run time (samsim_b200_set_tuning): the library carries two instantiations
// of the step kernel, samsim_step_kernel<false> (general path only) and samsim_step_kernel<true>.

// May this column take the merged forward pass in this step?  Everything here is a per-column, per-step decision.
__device__ __forceinline__ bool fast_path_ok(const Col& c, bool output_step, bool observable_after) {
  if (!(c.thermo_valid && c.pre.valid) || output_step || observable_after) return false;
  if (c.N_active < 3 || c.i == 1) return false;
  if (CFG.grav_flag != 2 || CFG.harmonic_flag != 2 || CFG.n_bgc != 0 || CFG.prescribe_flag == 2 || CFG.tank_flag == 2) return false;
  if (!(CFG.boundflux_flag == 1 || CFG.boundflux_flag == 2)) return false;
  if (CFG.testcase == 5 || (CFG.testcase >= 101 && CFG.testcase <= 105)) return false;  // hooks that edit the column / read S_bu
  // snow: a layer of its own (>= thick_min) or none at all; thin snow couples to layer 1 (S10, S17) -> general path
  const double ts = SCV(c, SC_THICK_SNOW), ms = SCV(c, SC_M_SNOW);
  if (!(ts >= CFG.thick_min || (ms <= 0.0 && ts < CFG.thick_min / 100.0))) return false;
  if (CFG.flood_flag > 1) {
    // S11: func_freeboard < 0 needs either m_snow > total buoyancy (mo_functions.f90:99) or a waterline in layer 1.
    // With m(1) + m_snow below the buoyancy of layers 2..Na (psi_s part only, backward-order sum, 1e-9 safety) the
    // waterline is in layer 2 or deeper and the freeboard is >= thick(1) > 0: no flooding, rigorously.
    const double snowmass = (CFG.freeboard_snow_flag == 0) ? ms : 0.0;
    if (!(c.m()[1] + snowmass < c.pre.A2 * (rho_l - rho_s) * (1.0 - 1e-9))) return false;
  }
  return true;
}

// One layer of S4 (volume fractions) + S5 (expulsion_flux, mass_transfer) + S7 for the forward pass.
// In: the layer's S4 values (m, S_abs, H_abs, thick, T, phi, S_bu = S_abs/m), its neighbours' S4 values, fl_m(k) = f0.
// Out: psi_* (psi_g after expulsion_flux), fl_m(k+1) = f1, m, S_abs, H_abs after the transfer.
//
// expulsion_flux only ever produces fl_m <= 0 (V_ex >= 0, mo_mass.f90:121-134: -V_ex*rho_l + fl_m(k) with fl_m(1) = 0, or
// -MAX(.., 0)), so of mass_transfer's four branches (mo_mass.f90:76-95) only `fl_m(k+1) < 0` (the layer loses its own
// brine) and `fl_m(k) < 0` (it receives the brine of the layer above) can be taken here: the layer BELOW is never read,
// and the forward pass needs no look-ahead.  (NaN fluxes take neither branch, exactly like the general routine.)
struct Expelled { double ps, pl, pg, f1, m_new, S, H; };
__device__ __forceinline__ Expelled expel_layer(int k, double phi_k, double thk, double m_k, double Sabs_k, double H_k, double T_k,
                                                double sbu_k, double f0, double T_km1, double SbuE_km1, double SabsE_km1) {
  Expelled e;
  double vex;
  expulsion(phi_k, thk, m_k, e.ps, e.pl, e.pg, vex);
  if (k == 1) {  // fl_m(k+1), mo_mass.f90:121-134
    e.f1 = -vex * rho_l;
  } else if (e.pg < SAMSIM_F32(0.001)) {
    e.f1 = -vex * rho_l + f0;
  } else {
    e.f1 = -f_max((vex - e.pg * thk) * rho_l, 0.0);
    e.pg = f_max((e.pg * thk - vex) / thk, 0.0);
  }
  e.m_new = m_k + e.f1 - f0;
  e.S = Sabs_k; e.H = H_k;
  if (e.f1 < 0.) {  // mo_mass.f90:82-84
    e.H = e.H + e.f1 * T_k * c_l;
    e.S = e.S + f_max(e.f1 * S_br_of(T_k, sbu_k), -e.S);
  }
  if (f0 < 0) {     // :89-92 (S_abs(k-1) is the value the transfer of layer k-1 left)
    e.H = e.H - f0 * T_km1 * c_l;
    e.S = e.S - f_max(f0 * S_br_of(T_km1, SbuE_km1), -SabsE_km1);
  }
  return e;
}

// S9 gas in the lowest layer (mo_grotz.f90:405-410) and S12 sub_turb_flux (mo_functions.f90:347-363) on layer N_active
__device__ __forceinline__ void bottom_layer_updates(Col& c, double pg, double thk, double T_Na, double& m_new, double& S, double& H) {
  const double T_bottom = SCV(c, SC_T_BOTTOM), S_bu_bottom = SCV(c, SC_S_BU_BOTTOM);
  if (pg > 0.0) {
    EVT(c, EV_GAS_REFILL);
    const double g2 = pg * thk * rho_l;
    m_new = m_new + g2;
    S = S + g2 * S_bu_bottom;
    H = H + g2 * c_l * T_bottom;
  }
  if (CFG.turb_flag == 2) {
    EVT(c, EV_TURB);
    const double turb = Turb_A * det_exp(Turb_B * (-density_of(T_bottom, S_bu_bottom) + density_of(T_Na, S / m_new))) * CFG.dt;
    S = S - turb * (S / m_new - S_bu_bottom);
  }
}

// ray(k) by the reference's forward sums (mo_grav_drain.f90:115-120, :128, :126-136) for one layer whose estimate can
// exceed ray_crit.  Out of line: the forward pass calls it for the few candidate layers only.
__device__ __noinline__ double exact_ray(const Col& c, int k, double sbr_k) {
  const View v = c;
  const int Na = c.N_active;
  const double bottom_h = c.pre.bottom_h;
  const double qb = bottom_h / c.pre.perm_Na;
  Lay q = v.w1();
  double hq = 0.0, ht = 0.0, hb = 0.0;
  SAMSIM_LOOP
  for (int kk = k; kk <= Na - 1; kk++) {
    const double tv = v.thick()[kk];
    hq = hq + q[kk];
    ht = ht + tv;
    if (kk > k) hb = hb + tv;
  }
  double hp = hq + qb;  // the estimate was > 0, so minval(perm(k:Na-1)) >= 1e-14 (:112) holds
  hp = (ht + bottom_h) / hp;
  double r = grav * rho_l * bbeta * (sbr_k - c.pre.S_br_Na) * (hb + bottom_h) * hp;
  r = r / (kappa_l * mu);
  return f_max(r, 0.0);
}
// Layer 1 of the Rayleigh estimate (layers >= 2 were prepared by backward_pass); stores thick(1)/perm(1) for exact_ray.
__device__ __noinline__ double ray_estimate_layer1(const Col& c, double pl, double thk, double sbr_1) {
  const View v = c;
  const double bottom_h = c.pre.bottom_h;
  const double qb = bottom_h / c.pre.perm_Na;
  const double pk = 1e-17 * det_pow(1000.0 * fabs(pl), 3.10);
  const double qk = thk / pk;
  v.w1()[1] = qk;
  const double mn = (c.N_active == 2) ? pk : f_min(c.pre.mn2, pk);
  const double hp = (mn < 1e-14) ? 0.0 : ((c.pre.st2 + thk) + bottom_h) / ((c.pre.sq2 + qk) + qb);
  double est = grav * rho_l * bbeta * (sbr_1 - c.pre.S_br_Na) * (c.pre.st2 + bottom_h) * hp;
  est = est / (kappa_l * mu);
  return (mn < 1e-14) ? 0.0 : f_max(est, 0.0);
}
// One draining layer (mo_grav_drain.f90:146-166): S_abs, H_abs of the layer, the accumulators, fl_up(k) (returned).
// Returns a negative value on STOP 21234.
__device__ __noinline__ double drain_layer(Col& c, double rk, double thk, double pl, double T_k, double sbr_k, double& S, double& H,
                                           double& run, double& heat_loss) {
  double flux = x_grav * (rk - ray_crit) * CFG.dt * thk;
  flux = f_min(flux, pl * rho_l * thk);
  S = S - flux * sbr_k;
  if (S < 0.0) { c.status = 21234; return -1.0; }
  SCV(c, SC_GRAV_TEMP) = SCV(c, SC_GRAV_TEMP) + flux * T_k;
  H = H - flux * c_l * T_k;
  heat_loss = heat_loss + flux * c_l * T_k;
  run = run + flux;
  return f_min(run, pl * rho_l * thk);
}

#ifndef SAMSIM_MERGE_HEAT
#define SAMSIM_MERGE_HEAT 1   // 1: sub_heat_fluxes' layer update rides along phase A of the forward pass; 0: it stays a sweep of its own
#endif

// S4 .. S17 of one step in one forward pass (see the block comment above).  Preconditions: fast_path_ok().
//
// Phase A (layers above the first draining layer kfirst): per iteration k the layer is expelled (E), its drain
// decision is taken (D), and layer k-1 gets its heat-flux update (Q) -- gravity drainage moves nothing above kfirst,
// so those layers are final.  Phase B (k >= kfirst, typically the warm bottom fifth of the column): E and D only;
// the drainage mass_transfer (which needs S_abs(k+1) after ITS drain) and the heat update of these layers follow in
// the reference's own order on the layers kfirst..N_active.  The loops touch nothing of `c`: every per-column scalar
// they need is a local, rare events are out-of-line calls, the minima of the health checks are sign flags.
__device__ __noinline__ void forward_pass(Col& c) {
  const View v = c;
  const int Na = c.N_active;
  const double dt = CFG.dt;
  const double T_bottom = SCV(c, SC_T_BOTTOM), S_bu_bottom = SCV(c, SC_S_BU_BOTTOM);
  const double cand = ray_crit * (1.0 - 1e-10);
  const bool merge_heat = SAMSIM_MERGE_HEAT;

  double temp1 = 0.0, temp2 = 0.0;             // energy check sums, mo_heat_fluxes.f90:269, :305
  double sum_before = 0.0, sum_after = 0.0;    // SUM(S_abs) of mo_grav_drain.f90:141 / :173
  double fbA = 0.0, fbG = 0.0, fbAs = 0.0, fbGs = 0.0;  // func_freeboard memo
  bool neg_ps = false, neg_S = false;          // MINVAL(psi_s) < 0 (S24), MINVAL(S_abs) < 0 (:198): only the sign is used
  const int ks = (c.fb.k_last >= 1 && c.fb.k_last < Na) ? c.fb.k_last : 0;
  int kfirst = 0;
  double run = 0.0, heat_loss = 0.0;
  double H_km1 = 0.0, hr_km1 = 0.0, fq_km1 = 0.0, rad = 0.0, flQ1 = 0.0;  // Q: layer k-1 waiting for its lower flux

  // ---- layer 1: the S4 getT (layers >= 2 keep T, phi of the S18 sweep: same inputs, same first-guess chain) ----
  double T_km1, SbuE_km1, SabsE_km1, f0;       // E: layer k-1's S4 values, its S_abs after the transfer, fl_m(k)
  {
    const double m_k = v.m()[1], Sabs_k = v.S_abs()[1], H_k = v.H_abs()[1], thk = v.thick()[1];
    const double sbu_k = Sabs_k / m_k;                 // S_bu(k) of S4 (:299)
    double T_k, phi_k = v.phi()[1];
    getT(H_k / m_k, sbu_k, v.T()[2], T_k, phi_k, c.status, c.ev1);
    v.T()[1] = T_k; v.phi()[1] = phi_k;
    // ---- E(1), D(1) peeled: layer 1 has no upper neighbour, makes its own Rayleigh estimate, and (when it does not
    //      drain) is final right away, so the surface energy balance can be evaluated before the loop ----
    Expelled e = expel_layer(1, phi_k, thk, m_k, Sabs_k, H_k, T_k, sbu_k, 0.0, 0.0, 0.0, 0.0);
    v.psi_s()[1] = e.ps; v.psi_l()[1] = e.pl; v.psi_g()[1] = e.pg; v.m()[1] = e.m_new;
    fbA = fbA + e.ps * thk;
    fbG = fbG + e.pg * thk;
    neg_ps = neg_ps || (e.ps < 0.0);
    const double SabsE_1 = e.S;
    const double sbr_1 = S_br_of(T_k, sbu_k);
    double rk = ray_estimate_layer1(c, e.pl, thk, sbr_1);
    if (rk > cand) rk = exact_ray(c, 1, sbr_1);
    sum_before = sum_before + e.S;
    if (rk > ray_crit && e.ps > 0.001 && e.S / e.m_new > 0.1 && sbr_1 > S_br_of(v.T()[2], v.S_abs()[2] / v.m()[2])) {
      kfirst = 1;
      EVT(c, EV_GRAV_DRAINED);
      const double up = drain_layer(c, rk, thk, e.pl, T_k, sbr_1, e.S, e.H, run, heat_loss);
      if (up < 0.0) return;
      sum_after = 0.0 + e.S;
      v.S_abs()[1] = e.S; v.H_abs()[1] = e.H;
      v.S_bu()[1] = SabsE_1 / e.m_new;  // S7
      v.fl_m()[1] = 0.0; v.fl_m()[2] = up;
    } else {
      v.S_abs()[1] = e.S;
      neg_S = neg_S || (e.S < 0.0);
      if (merge_heat) {  // surface energy balance, mo_heat_fluxes.f90:77-195 (layer 1 is final)
        double fl_rad_Na;
        const SurfIn in = {e.ps, e.pl, e.pg, thk, T_k, e.S, e.m_new, 0.0, 0.0, v.fl_Q()[1]};
        flQ1 = heat_surface(c, in, fl_rad_Na);
        fq_km1 = flQ1;
        rad = fl_rad_Na * dt;
        H_km1 = e.H;
        hr_km1 = thk / (2.0 * (e.ps * k_s + e.pl * k_l + e.pg * 0.0));  // half resistance of layer 1, sub_fl_Q
      } else {
        v.H_abs()[1] = e.H;
      }
    }
    T_km1 = T_k; SbuE_km1 = sbu_k; SabsE_km1 = SabsE_1; f0 = e.f1;
  }

  // =============================== phase A: k = 2 .. kfirst (or N_active) ===============================
  int k = 2;
  if (!kfirst) {
    SAMSIM_LOOP
    for (; k <= Na; k++) {
      if (k + SAMSIM_PF <= Na) {
        const int kp = k + SAMSIM_PF;
        v.T().prefetch(kp); v.phi().prefetch(kp); v.m().prefetch(kp); v.thick().prefetch(kp); v.S_abs().prefetch(kp);
        v.H_abs().prefetch(kp); v.ray().prefetch(kp);
      }
      // ---- the layer's S4 values: T, phi of the S18 sweep, S_bu = S_abs/m (:299) ----
      const double m_k = v.m()[k], Sabs_k = v.S_abs()[k], H_k = v.H_abs()[k], thk = v.thick()[k], T_k = v.T()[k], phi_k = v.phi()[k];
      const double sbu_k = Sabs_k / m_k;
      // ---- E(k) ----
      Expelled e = expel_layer(k, phi_k, thk, m_k, Sabs_k, H_k, T_k, sbu_k, f0, T_km1, SbuE_km1, SabsE_km1);
      v.psi_s()[k] = e.ps; v.psi_l()[k] = e.pl; v.psi_g()[k] = e.pg;
      fbA = fbA + e.ps * thk;
      fbG = fbG + e.pg * thk;
      if (ks && k > ks) { fbAs = fbAs + e.ps * thk; fbGs = fbGs + e.pg * thk; }
      neg_ps = neg_ps || (e.ps < 0.0);
      const double SabsE_k = e.S;
      if (k == Na) bottom_layer_updates(c, e.pg, thk, T_k, e.m_new, e.S, e.H);
      v.m()[k] = e.m_new;
      // ---- Q(k-1): heat update of the layer above (final: nothing drains above kfirst) ----
      double hr_k = 0.0;
      if (merge_heat) {
        hr_k = thk / (2.0 * (e.ps * k_s + e.pl * k_l + 0.0 * 0.0));  // half resistance, sub_fl_Q
        const double fq_k = (T_k - T_km1) / (hr_km1 + hr_k);          // fl_Q(k), :272-274
        double Hh = H_km1;
        temp1 = temp1 + Hh;                  // :269
        Hh = Hh + (fq_k - fq_km1) * dt;      // :277-279
        Hh = Hh + rad;                       // :282-285 (sic)
        v.H_abs()[k - 1] = Hh;
        temp2 = temp2 + Hh;
        fq_km1 = fq_k;
      }
      // ---- D(k): does this layer drain?  (mo_grav_drain.f90:145) ----
      bool drains = false;
      if (k < Na) {
        double rk = v.ray()[k];
        if (rk > cand) {
          const double sbr_k = S_br_of(T_k, sbu_k);
          rk = exact_ray(c, k, sbr_k);
          if (rk > ray_crit && e.ps > 0.001 && e.S / e.m_new > 0.1 && sbr_k > S_br_of(v.T()[k + 1], v.S_abs()[k + 1] / v.m()[k + 1])) {
            // first draining layer: the layers from here on are settled in phase B
            drains = true;
            kfirst = k;
            EVT(c, EV_GRAV_DRAINED);
            const double prefix = sum_before;   // SUM(S_abs) before (:141) and after (:173) share the terms 1..kfirst-1
            sum_before = prefix + e.S;
            const double up = drain_layer(c, rk, thk, e.pl, T_k, sbr_k, e.S, e.H, run, heat_loss);
            if (up < 0.0) return;
            sum_after = prefix + e.S;
            v.S_abs()[k] = e.S; v.H_abs()[k] = e.H;
            v.S_bu()[k] = SabsE_k / e.m_new;                          // S7 of layer k
            v.S_bu()[k - 1] = v.S_abs()[k - 1] / v.m()[k - 1];        // S7 of layer k-1 (it did not drain: S_abs is its S5 value)
            v.fl_m()[k] = 0.0;
            v.fl_m()[k + 1] = up;
          }
        }
      }
      if (!drains) {
        if (k < Na) sum_before = sum_before + e.S;
        v.S_abs()[k] = e.S;
        neg_S = neg_S || (e.S < 0.0);
        if (!merge_heat) v.H_abs()[k] = e.H;
      }
      // ---- shift the window ----
      T_km1 = T_k; SbuE_km1 = sbu_k; SabsE_km1 = SabsE_k; H_km1 = e.H; hr_km1 = hr_k;
      f0 = e.f1;
      if (drains) { k++; break; }
    }
  }

  const double fl_q_bottom = SCV(c, SC_FL_Q_BOTTOM);
  if (!kfirst) {
    // nothing drained: SUM(S_abs) before = after (:141, :173), no transfer; layer N_active awaits its heat update
    const double S_Na = v.S_abs()[Na];  // after S9 / S12
    sum_before = sum_before + S_Na;
    SCV(c, SC_GRAV_SALT) = SCV(c, SC_GRAV_SALT) + sum_before;
    SCV(c, SC_GRAV_SALT) = SCV(c, SC_GRAV_SALT) - sum_before;
    SCV(c, SC_GRAV_DRAIN) = SCV(c, SC_GRAV_DRAIN) + run;                                // :190 (run = 0)
    double H_Na = H_km1;
    if (CFG.grav_heat_flag == 2) H_Na = H_Na + heat_loss - run * c_l * T_bottom;       // :193-195 (adds 0 - 0)
    if (neg_S) c.status = 1337;                                                          // :198
    if (merge_heat) {
      temp1 = temp1 + H_Na;
      H_Na = H_Na + (fl_q_bottom - fq_km1) * dt;
      H_Na = H_Na + rad;
      v.H_abs()[Na] = H_Na;
      temp2 = temp2 + H_Na;
    } else {
      v.H_abs()[Na] = H_Na;
    }
  } else {
    // =============================== phase B: k = kfirst+1 .. N_active, E and D only ===============================
    SAMSIM_LOOP
    for (; k <= Na; k++) {
      if (k + SAMSIM_PF <= Na) {
        const int kp = k + SAMSIM_PF;
        v.T().prefetch(kp); v.phi().prefetch(kp); v.m().prefetch(kp); v.thick().prefetch(kp); v.S_abs().prefetch(kp);
        v.H_abs().prefetch(kp); v.ray().prefetch(kp);
      }
      const double m_k = v.m()[k], Sabs_k = v.S_abs()[k], H_k = v.H_abs()[k], thk = v.thick()[k], T_k = v.T()[k], phi_k = v.phi()[k];
      const double sbu_k = Sabs_k / m_k;
      Expelled e = expel_layer(k, phi_k, thk, m_k, Sabs_k, H_k, T_k, sbu_k, f0, T_km1, SbuE_km1, SabsE_km1);
      v.psi_s()[k] = e.ps; v.psi_l()[k] = e.pl; v.psi_g()[k] = e.pg;
      fbA = fbA + e.ps * thk;
      fbG = fbG + e.pg * thk;
      if (ks && k > ks) { fbAs = fbAs + e.ps * thk; fbGs = fbGs + e.pg * thk; }
      neg_ps = neg_ps || (e.ps < 0.0);
      const double SabsE_k = e.S;
      v.S_bu()[k] = e.S / e.m_new;  // S7
      if (k == Na) bottom_layer_updates(c, e.pg, thk, T_k, e.m_new, e.S, e.H);
      v.m()[k] = e.m_new;
      double up_k = run;
      if (k < Na) {
        sum_before = sum_before + e.S;
        double rk = v.ray()[k];
        if (rk > cand) {
          const double sbr_k = S_br_of(T_k, sbu_k);
          rk = exact_ray(c, k, sbr_k);
          if (rk > ray_crit && e.ps > 0.001 && e.S / e.m_new > 0.1 && sbr_k > S_br_of(v.T()[k + 1], v.S_abs()[k + 1] / v.m()[k + 1])) {
            up_k = drain_layer(c, rk, thk, e.pl, T_k, sbr_k, e.S, e.H, run, heat_loss);
            if (up_k < 0.0) return;
          }
        }
        sum_after = sum_after + e.S;
      }
      v.S_abs()[k] = e.S; v.H_abs()[k] = e.H;
      v.fl_m()[k + 1] = up_k;  // fl_m(k+1) = fl_up(k); for k = N_active that is the running sum (:162-164, :177)
      T_km1 = T_k; SbuE_km1 = sbu_k; SabsE_km1 = SabsE_k;
      f0 = e.f1;
    }
    const double S_Na = v.S_abs()[Na];
    sum_before = sum_before + S_Na;
    sum_after = sum_after + S_Na;
    SCV(c, SC_GRAV_SALT) = SCV(c, SC_GRAV_SALT) + sum_before;  // :141
    SCV(c, SC_GRAV_SALT) = SCV(c, SC_GRAV_SALT) - sum_after;   // :173
    mass_transfer(c, v.fl_m(), v.S_bu(), kfirst);               // :188
    SCV(c, SC_GRAV_DRAIN) = SCV(c, SC_GRAV_DRAIN) + run;        // :190
    if (CFG.grav_heat_flag == 2) v.H_abs()[Na] = v.H_abs()[Na] + heat_loss - run * c_l * T_bottom;  // :193-195
    SAMSIM_LOOP
    for (int kk = kfirst; kk <= Na; kk++) neg_S = neg_S || (v.S_abs()[kk] < 0.0);
    if (neg_S) c.status = 1337;                                  // :198
    if (merge_heat) {
      // ---- heat update of layers kfirst .. N_active (mo_heat_fluxes.f90:272-285) ----
      int j = kfirst;
      double T_j = v.T()[j];
      double hr_j;
      if (j == 1) {
        double fl_rad_Na;
        const SurfIn in = {v.psi_s()[1], v.psi_l()[1], v.psi_g()[1], v.thick()[1], v.T()[1], v.S_abs()[1], v.m()[1], 0.0, 0.0, v.fl_Q()[1]};
        flQ1 = heat_surface(c, in, fl_rad_Na);
        fq_km1 = flQ1;
        rad = fl_rad_Na * dt;
        hr_j = v.thick()[1] / (2.0 * (v.psi_s()[1] * k_s + v.psi_l()[1] * k_l + v.psi_g()[1] * 0.0));
      } else {
        hr_j = hr_km1;  // layer kfirst's half resistance and the flux into it were evaluated with Q(kfirst-1)
      }
      SAMSIM_LOOP
      for (; j <= Na; j++) {
        double fq_jp1, hr_n = 0.0, T_n = 0.0;
        if (j < Na) {
          const double ps_n = v.psi_s()[j + 1], pl_n = v.psi_l()[j + 1], th_n = v.thick()[j + 1];
          T_n = v.T()[j + 1];
          hr_n = th_n / (2.0 * (ps_n * k_s + pl_n * k_l + 0.0 * 0.0));
          fq_jp1 = (T_n - T_j) / (hr_j + hr_n);
        } else {
          fq_jp1 = fl_q_bottom;
        }
        double Hh = v.H_abs()[j];
        temp1 = temp1 + Hh;
        Hh = Hh + (fq_jp1 - fq_km1) * dt;
        Hh = Hh + rad;
        v.H_abs()[j] = Hh;
        temp2 = temp2 + Hh;
        fq_km1 = fq_jp1; hr_j = hr_n; T_j = T_n;
      }
    }
  }

  c.fb.tot_valid = true; c.fb.t1 = v.thick()[1]; c.fb.A = fbA; c.fb.G = fbG;
  c.fb.suf_valid = (ks != 0); c.fb.ks = ks; c.fb.As = fbAs; c.fb.Gs = fbGs;
  c.fb.res_valid = false;
  c.min_psi_s = neg_ps ? -1.0 : 1.0;  // S24 reads the sign only

  if (!merge_heat) {
    if (c.status == 0) heat_fluxes(c);  // S17 as a sweep of its own
    return;
  }
  v.fl_Q()[1] = flQ1;
  v.fl_Q()[Na + 1] = fl_q_bottom;  // :262
  temp1 = temp1 + SCV(c, SC_H_ABS_SNOW);
  SAMSIM_LOOP
  for (int kk = 1; kk <= Na; kk++) temp1 = temp1 + rad;  // :284
  if (SCV(c, SC_THICK_SNOW) >= CFG.thick_min) {  // :296-299 (thin snow never takes this path)
    const double fl_q_snow = SCV(c, SC_FL_Q_SNOW);
    SCV(c, SC_H_ABS_SNOW) = SCV(c, SC_H_ABS_SNOW) + (flQ1 - fl_q_snow) * dt;
    temp1 = temp1 + fl_q_bottom * dt - fl_q_snow * dt;
  } else {
    temp1 = temp1 + fl_q_bottom * dt - flQ1 * dt;  // :302
  }
  temp2 = temp2 + SCV(c, SC_H_ABS_SNOW);
  if (c.status == 0 && fabs((temp1 - temp2) / dt) > 0.00001) c.status = 431;  // :307-310
}

template <bool TWO_PASS>
__device__ __noinline__ void column_step(Col& c, const Forcing& f, bool want_diag, const SnapOut& snap) {
  const View v = c;
  const double dt = CFG.dt;
  const int N = CFG.Nlayer;
  c.i = c.i + 1;
  c.want_state = want_diag;
  const bool output_step = (c.n_time_out == CFG.i_time_out || c.i == 1);

  if (c.status == 0) {  // ===== phase 0 =====
  // ---- S0 :192-223 (only observable at S8 or through get_scalar after the launch) ----
  if (output_step || want_diag) vital_signs(c);

  // ---- S1 forcing :229-246 ----
  if (CFG.atmoflux_flag == 2) {
    if (c.time > time_input(c.time_counter)) c.time_counter = c.time_counter + 1;
    const int tc = c.time_counter;
    c.ftime1 = time_input(tc);
    c.fsw1 = forcing_rec(f, 0, tc);
    c.flw1 = forcing_rec(f, 1, tc);
    if (c.time == c.ftime1) {
      SCV(c, SC_T2M) = forcing_rec(f, 2, tc);
      SCV(c, SC_LIQUID_PRECIP) = forcing_rec(f, 3, tc);
      c.ftime0 = 0.0; c.fsw0 = 0.0; c.flw0 = 0.0;
    } else {
      c.ftime0 = time_input(tc - 1);
      c.fsw0 = forcing_rec(f, 0, tc - 1);
      c.flw0 = forcing_rec(f, 1, tc - 1);
      const double temp = (c.time - c.ftime0) / (c.ftime1 - c.ftime0);
      SCV(c, SC_T2M) = (1.0 - temp) * forcing_rec(f, 2, tc - 1) + temp * forcing_rec(f, 2, tc);
      SCV(c, SC_LIQUID_PRECIP) = (1.0 - temp) * forcing_rec(f, 3, tc - 1) + temp * forcing_rec(f, 3, tc);
    }
  }
  long long lab_idx = 0;
  if (CFG.boundflux_flag == 3 && CFG.lab_snow_flag == 1) {  // :244-246
    lab_idx = (long long)floor(1 + c.time / dt);
    SCV(c, SC_SOLID_PRECIP) = lab_rec(f, 1, lab_idx);
  }

  // ---- S2 snow fall :251-265 ----
  {
    const double lp = SCV(c, SC_LIQUID_PRECIP), sp = SCV(c, SC_SOLID_PRECIP);
    if (f_max(lp, sp) > 0.0 && (CFG.precip_flag == 1 || CFG.precip_flag == 0)) {
      const bool have_solid = (CFG.precip_flag == 0);
      if (c.N_active > 1) {
        EVT(c, EV_SNOW_PRECIP);
        snow_precip(c, dt, lp, SCV(c, SC_T2M), have_solid, sp);
      } else if (c.N_active == 1) {
        EVT(c, EV_SNOW_PRECIP_0);
        double H1 = v.H_abs()[1], S1 = v.S_abs()[1];
        snow_precip_0(H1, S1, v.m()[1], v.T()[1], dt, lp, SCV(c, SC_T2M), have_solid, sp);
        v.H_abs()[1] = H1; v.S_abs()[1] = S1;
      }
    }
  }

  // ---- S3 snow thermodynamics :273-292 ----
  snow_block(c);

  }
  SAMSIM_PHASE_SYNC();
  // Two-pass step (forward_pass / backward_pass above) or the general sub-step-by-sub-step path?  Decided per column
  // after S3: the snow state and m(1) are final for this step's S10 / S11 decisions.
  const bool next_step_outputs_pre = ((output_step ? 0 : c.n_time_out + 1) == CFG.i_time_out);
  const bool fast = TWO_PASS && (c.status == 0) && fast_path_ok(c, output_step, want_diag || next_step_outputs_pre);
  if (c.status == 0 && !fast) {  // ===== phase 1 =====
  // ---- S4 :298-307, S5 :312-321, S7 :333-335 ----
  // S4's getT sweep is the same computation as S18's (S_bu = S_abs/m, H = H_abs/m, first guess chained from the layer
  // below, T_bottom at N_active).  When nothing touched m, S_abs, H_abs of layers 2..N_active since the S18 sweep of
  // the previous step (c.thermo_valid), it would return the same T, phi and is skipped; otherwise (first step of a
  // launch, after flushing or a layer event) it is run as that sweep.  Either way the volume fractions (Expulsion),
  // expulsion_flux, mass_transfer and S7 then run as ONE forward pass with fl_m, V_ex, S_br in registers; layer 1
  // (snow, precipitation, melt water) is always recomputed there.
  if (!c.thermo_valid) backward_pass<false>(c, false, false);
  fused_thermo_expulsion(c);

  }
  SAMSIM_PHASE_SYNC();
  if (c.status == 0) {  // ===== phase 2 =====
  c.fb_x = 0.0;
  // ---- S8 output :340-398 ----
  if (output_step) {
    SCV(c, SC_FREEBOARD) = (c.N_active > 1) ? freeboard_of(c) : 0.0;
    if (CFG.grav_flag == 2) {
      if (SCV(c, SC_GRAV_DRAIN) == 0.0) SCV(c, SC_GRAV_TEMP) = 0.0;
      else SCV(c, SC_GRAV_TEMP) = SCV(c, SC_GRAV_TEMP) / SCV(c, SC_GRAV_DRAIN);
      SCV(c, SC_GRAV_SALT) = SCV(c, SC_GRAV_SALT) / CFG.time_out;
      SCV(c, SC_GRAV_DRAIN) = SCV(c, SC_GRAV_DRAIN) / CFG.time_out;
    }
    write_snapshot(c, snap);
    SCV(c, SC_GRAV_DRAIN) = 0.0; SCV(c, SC_GRAV_SALT) = 0.0; SCV(c, SC_GRAV_TEMP) = 0.0;
    SCV(c, SC_MTO1) = 0.0; SCV(c, SC_MTO2) = 0.0; SCV(c, SC_MTO3) = 0.0;
    c.n_time_out = 0;
  } else {
    c.n_time_out = c.n_time_out + 1;
  }

  }
  SAMSIM_PHASE_SYNC();
  if (c.status == 0 && !fast) {  // ===== phase 3 =====
  // ---- S9 gas in the lowest layer :405-410 ----
  {
    const int Na = c.N_active;
    const double pg = v.psi_g()[Na];
    if (pg > 0.0) {
      EVT(c, EV_GAS_REFILL);
      const double temp2 = pg * v.thick()[Na] * rho_l;
      c.fb.res_valid = false;
      v.m()[Na] = v.m()[Na] + temp2;
      v.S_abs()[Na] = v.S_abs()[Na] + temp2 * SCV(c, SC_S_BU_BOTTOM);
      v.H_abs()[Na] = v.H_abs()[Na] + temp2 * c_l * SCV(c, SC_T_BOTTOM);
    }
  }

  // ---- S10 thin snow coupling :418-420 ----
  if (SCV(c, SC_M_SNOW) > 0.0 && SCV(c, SC_THICK_SNOW) < CFG.thick_min) {
    double H1 = v.H_abs()[1], phi1 = v.phi()[1], T1 = v.T()[1];
    snow_coupling(c, H1, phi1, T1, v.m()[1], v.S_bu()[1]);
    v.H_abs()[1] = H1; v.phi()[1] = phi1; v.T()[1] = T1;
    }

  // ---- S11 flooding :428-445 ----
  if (c.N_active > 1 && CFG.flood_flag > 1) {
    SCV(c, SC_FREEBOARD) = freeboard_of(c);
    if (SCV(c, SC_FREEBOARD) < 0.0) {
      if (CFG.flood_flag == 2) { flood(c); fb_reset(c); }
      else if (CFG.flood_flag == 3 && SCV(c, SC_FREEBOARD) < neg_free) { flood_simple(c); fb_reset(c); }
    }
  }

  // ---- S12 turbulence (sub_turb_flux, mo_functions.f90:347-363) :450-457 ----
  if (CFG.turb_flag == 2) {
    EVT(c, EV_TURB);
    const int Na = c.N_active;
    const double S = v.S_abs()[Na], mNa = v.m()[Na];
    const double turb = Turb_A * det_exp(Turb_B * (-density_of(SCV(c, SC_T_BOTTOM), SCV(c, SC_S_BU_BOTTOM)) + density_of(v.T()[Na], S / mNa))) * dt;
    v.S_abs()[Na] = S - turb * (S / mNa - SCV(c, SC_S_BU_BOTTOM));
    for (int q = 0; q < CFG.n_bgc; q++) {  // mo_functions.f90:357-359
      const double b = v.bgc(q)[Na];
      v.bgc(q)[Na] = b - turb * (b / mNa - SCV(c, SC_BGC_BOTTOM1 + q));
    }
  }

  }
  SAMSIM_PHASE_SYNC();
  if (TWO_PASS) {
    if (c.status == 0 && fast) {  // ===== phase 4, two-pass step: S4 .. S17 in one forward pass =====
      EVT(c, EV_TWO_PASS_STEP);
      testcase_hooks(c, f);  // S15: these testcases' hooks depend on the clock only (fast_path_ok), so they commute with S4-S13
      forward_pass(c);
    }
  }
  if (c.status == 0 && !fast) {  // ===== phase 4 =====
  // ---- S13 gravity drainage :463-477 ----
  if (CFG.grav_flag == 2 && c.N_active > 1) {
    // ray(1:N-1) is observable through the S8 record of the next step (n_time_out was already advanced by S8 above)
    // and through get_array after the launch; otherwise only layers that can drain need their exact value
    const bool next_step_outputs = (c.n_time_out == CFG.i_time_out);
    grav_drain(c, c.want_state || next_step_outputs);
  }
  else if (CFG.grav_flag == 3 && c.N_active > 1) { EVT(c, EV_GRAV_DRAIN_SIMPLE); grav_drain_simple(c); }

  // ---- S14 prescribed salinity profile :482-497 (prescribe_flag 2) ----
  if (CFG.prescribe_flag == 2) {
    EVT(c, EV_PRESCRIBE);
    const int Na = c.N_active;
    const double Sb = SCV(c, SC_S_BU_BOTTOM);
    int k = Na;
    while (k > 1 && sum_fwd(v.thick(), k, Na) < 0.15) {
      v.S_bu()[k] = Sb - sum_fwd(v.thick(), k, Na) / 0.15 * (Sb - 4.0);
      k = k - 1;
    }
    while (k > 1 && sum_fwd(v.thick(), k, Na) >= 0.15) {
      v.S_bu()[k] = 4.0 - 4.0 * (sum_fwd(v.thick(), k, Na) - 0.15) / (sum_fwd(v.thick(), 1, Na) - 0.15);
      k = k - 1;
      v.S_bu()[1] = 0.0;
    }
    v.S_bu()[Na] = Sb;
    SAMSIM_LOOP
    for (int kk = 1; kk <= N; kk++) v.S_abs()[kk] = v.S_bu()[kk] * v.m()[kk];  // S_abs = S_bu*m, whole arrays
  }

  }
  SAMSIM_PHASE_SYNC();
  if (c.status == 0 && !fast) {  // ===== phase 5 =====
  // ---- S15 testcase hooks :503-563 ----
  testcase_hooks(c, f);

  // ---- S16 tank :573-578 ----
  if (CFG.tank_flag == 2) {
    EVT(c, EV_TANK);
    SCV(c, SC_S_BU_BOTTOM) = (SCV(c, SC_S_TOTAL) - sum_fwd(v.S_abs(), 1, c.N_active)) / (CFG.m_total - sum_fwd(v.m(), 1, c.N_active));
    if (CFG.n_bgc) {  // :575-577 (sic: every tracer gets the value computed from tracer 1)
      const double vb = (SCV(c, SC_BGC_TOTAL1) - sum_fwd(v.bgc(0), 1, c.N_active)) / (CFG.m_total - sum_fwd(v.m(), 1, c.N_active));
      for (int q = 0; q < CFG.n_bgc; q++) SCV(c, SC_BGC_BOTTOM1 + q) = vb;
    }
  }

  // ---- S17 heat fluxes :584 ----
  heat_fluxes(c);

  }
  SAMSIM_PHASE_SYNC();
  if (c.status == 0) {  // ===== phase 6 =====
  // ---- S18 second backward sweep :592-598 (psi_* are NOT refreshed) ----
  {
    // Prepare the next step's merged forward pass unless ray must stay as fl_grav_drain left it (observable after
    // the launch or in the next step's S8 record).  S_bu is only observable after the launch.
    const bool next_step_outputs = (c.n_time_out == CFG.i_time_out);
    const bool prepare = TWO_PASS && !(c.want_state || next_step_outputs) && c.N_active >= 3 && CFG.grav_flag == 2 &&
                         CFG.harmonic_flag == 2 && CFG.n_bgc == 0;
    backward_pass<TWO_PASS>(c, prepare, c.want_state || SAMSIM_ALWAYS_STORE_S_BU);
  }

  }
  SAMSIM_PHASE_SYNC();
  if (c.status == 0) {  // ===== phase 7 =====
  // ---- S19 snow thermodynamics #2 :600-625 ----
  SCV(c, SC_MELT_THICK_SNOW_OLD) = SCV(c, SC_MELT_THICK_SNOW);
  snow_block(c);
  SCV(c, SC_MELT_THICK_SNOW) = SCV(c, SC_MELT_THICK_SNOW_OLD) + SCV(c, SC_MELT_THICK_SNOW);

  // ---- S20 flushing preparations :632-664 ----
  if (c.N_active > 1 && CFG.flush_flag > 2 && (CFG.boundflux_flag == 2 || CFG.boundflux_flag == 3)) {
    SCV(c, SC_T_FREEZE) = T_freeze_of(v.S_abs()[1] / v.m()[1], CFG.salt_flag);
    SCV(c, SC_MELT_THICK) = 0.0;
    if (freeboard_of(c) > 0.0000000000001) {
      const double ps1 = v.psi_s()[1];
      const double T_drive = (CFG.boundflux_flag == 2) ? SCV(c, SC_T_TOP) : SCV(c, SC_T2M);
      if (ps1 < psi_s_top_min || T_drive >= SCV(c, SC_T_FREEZE)) {
        double th1 = v.thick()[1];
        EVT(c, EV_MELT_THICK);
        if (melt_thick_of(v.psi_l()[1], ps1, v.psi_g()[1], v.T()[1], SCV(c, SC_T_FREEZE), T_drive, v.fl_Q()[1], SCV(c, SC_THICK_SNOW), dt,
                          SCV(c, SC_MELT_THICK), th1, CFG.thick_min)) EVT(c, EV_MELT_THICK_GAS);
        if (CFG.boundflux_flag == 3) SCV(c, SC_MELT_THICK) = f_max(SCV(c, SC_MELT_THICK), 0.0);
        if (SCV(c, SC_THICK_SNOW) >= CFG.thick_min / 100.0 && SCV(c, SC_MELT_THICK) > 0.00000000001 && SCV(c, SC_MELT_THICK_SNOW) == 0.0) {
          double H1 = v.H_abs()[1], m1 = v.m()[1];
          if (melt_snow(SCV(c, SC_MELT_THICK), th1, SCV(c, SC_THICK_SNOW), H1, SCV(c, SC_H_ABS_SNOW), m1, SCV(c, SC_M_SNOW), SCV(c, SC_PSI_G_SNOW)))
            EVT(c, EV_MELT_SNOW_ALL);
          else
            EVT(c, EV_MELT_SNOW_PART);
          v.H_abs()[1] = H1; v.m()[1] = m1;
        }
        v.thick()[1] = th1;
      }
    }
  }

  // ---- S21 flushing :670-737 ----
  SCV(c, SC_FREEBOARD) = freeboard_of(c);
  SCV(c, SC_MTO1) = SCV(c, SC_MTO1) + SCV(c, SC_MELT_THICK);
  SCV(c, SC_MTO2) = SCV(c, SC_MTO2) + SCV(c, SC_MELT_THICK_SNOW);
  SCV(c, SC_MELT_THICK) = SCV(c, SC_MELT_THICK) + SCV(c, SC_MELT_THICK_SNOW);
  if (SCV(c, SC_MELT_THICK_SNOW) > 0.0) {  // :677-685
    EVT(c, EV_SNOW_MELTWATER_TO_ICE);
    const double mts = SCV(c, SC_MELT_THICK_SNOW), T_snow = SCV(c, SC_T_SNOW);
    const double H1 = v.H_abs()[1] + mts * rho_l * c_l * T_snow;
    const double S1 = v.S_abs()[1] + mts * rho_l * S_br_of(T_snow, SCV(c, SC_S_ABS_SNOW) / SCV(c, SC_M_SNOW));
    const double m1 = v.m()[1] + mts * rho_l;
    v.H_abs()[1] = H1; v.S_abs()[1] = S1;
    v.thick()[1] = v.thick()[1] + mts;
    v.m()[1] = m1;
    v.S_bu()[1] = S1 / m1;
  }
  // flush_v/h: old = cur; cur = 0; [flush3 fills 1..N_active]; cur = cur + old  (:697-701, :736-737).
  // Without flush3 that is the identity; with it, new + old.  w-arrays hold the old values.
  if (c.N_active > 1 && SCV(c, SC_FREEBOARD) > 0.001) {
    if (CFG.flush_flag == 4) {  // :704-713
      const double mt = SCV(c, SC_MELT_THICK);
      if (mt > 0.000000000001 && c.N_active > 2) {
        EVT(c, EV_FLUSH_INLINE);
        const double m1 = v.m()[1];
        v.H_abs()[1] = v.H_abs()[1] - mt * rho_l * c_l * v.T()[1];
        v.S_abs()[1] = v.S_abs()[1] * (1.0 - (mt * rho_l) / m1);
        v.thick()[1] = v.thick()[1] - mt;
        v.m()[1] = m1 - mt * rho_l;
      }
    } else if (CFG.flush_flag == 5) {  // :715-728
      if (SCV(c, SC_MELT_THICK) > 0.000000000001 && c.N_active > 2 && SCV(c, SC_FREEBOARD) > 0.0) {
        SCV(c, SC_FREEBOARD) = freeboard_of(c);
        if (CFG.n_bgc == 0) {
          flush3_fused(c);  // adds this step's flush_v / flush_h to the accumulated arrays itself
        } else {
          const int Na = c.N_active;
          Lay old_v = v.V_ex(), old_h = v.S_br();  // both dead after S13
          SAMSIM_LOOP
          for (int k = 1; k <= Na; k++) { old_v[k] = v.flush_v()[k]; old_h[k] = v.flush_h()[k]; }
          flush3(c);
          SAMSIM_LOOP
          for (int k = 1; k <= Na; k++) { v.flush_v()[k] = v.flush_v()[k] + old_v[k]; v.flush_h()[k] = v.flush_h()[k] + old_h[k]; }
        }
        c.thermo_valid = false; c.pre.valid = false;
            }
    } else if (CFG.flush_flag == 6) {  // :729-733
      if (SCV(c, SC_MELT_THICK) > 0.000000000001 && c.N_active > 2 && SCV(c, SC_THICK_SNOW) < CFG.thick_0) {
        flush4(c);
        c.thermo_valid = false; c.pre.valid = false;
            }
    }
  }

  // ---- S22 tracer advection :742-747 ----
  if (CFG.n_bgc) bgc_advection(c);

  }
  SAMSIM_PHASE_SYNC();
  if (c.status == 0) {  // ===== phase 8 =====
  // ---- S23 layer dynamics :755-795 ----
  if (c.N_active > 1) {
    const int Na = c.N_active;
    const double r1 = v.thick()[1] / CFG.thick_0;
    if (v.phi()[Na] > psi_s_min || v.phi()[Na - 1] <= psi_s_min / 2.0 || r1 > 1.5 || r1 < 0.5) {
      layer_dynamics(c);
      c.thermo_valid = false; c.pre.valid = false;
      fb_reset(c);
        }
    const int Nb = c.N_active;
    if (Nb < N && v.thick()[(Nb + 1 < N) ? Nb + 1 : N] == 0) {  // :772-783 scrub
      EVT(c, EV_SCRUB);
      v.T()[Nb + 1] = SCV(c, SC_T_BOTTOM);
      v.S_bu()[Nb + 1] = SCV(c, SC_S_BU_BOTTOM);
      v.psi_l()[Nb + 1] = 1.0;
      v.psi_s()[Nb + 1] = 0.0;
      for (int q = 0; q < CFG.n_bgc; q++) v.bgc(q)[Nb + 1] = 0.0;  // :778-780
    }
  } else {
    if (v.phi()[1] > psi_s_min) { layer_dynamics(c); c.thermo_valid = false; c.pre.valid = false; fb_reset(c); }
    }

  // ---- S24 timestep + health check :802-819 ----
  c.time = c.time + dt;
  {
    const int Na = c.N_active;
    double mn, ms;
    if (c.thermo_valid) {
      // nothing touched psi_s(1:N_active) since S4, nor S_abs(2:N_active) since S18, and N_active is unchanged:
      // the minima gathered by those sweeps are the MINVALs of :808 and :812
      mn = c.min_psi_s;
      ms = f_min(v.S_abs()[1], c.min_S_abs_2);
    } else {
      mn = v.psi_s()[1]; ms = v.S_abs()[1];
      SAMSIM_LOOP
      for (int k = 2; k <= Na; k++) { mn = f_min(mn, v.psi_s()[k]); ms = f_min(ms, v.S_abs()[k]); }
    }
    if (mn < 0.0) {
      c.status = 1337;
    } else if (ms < 0.0) {
      EVT(c, EV_SALT_CLAMP);
      SAMSIM_LOOP
      for (int k = 1; k <= Na; k++) v.S_abs()[k] = f_max(v.S_abs()[k], 0.0);
      c.thermo_valid = false; c.pre.valid = false;
    }
  }
  }
  SAMSIM_PHASE_SYNC();
}

}  // namespace samsim
