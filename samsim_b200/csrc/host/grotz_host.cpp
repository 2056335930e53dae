// grotz_host.cpp -- C++ host side above the C ABI (include/samsim_b200_host.h).
//
// Mirrors the parts of the reference that stay on the host: init(testcase) (mo_init.f90), sub_input
// (mo_functions.f90:304-327), output_begin / output_settings / output (mo_output.f90) and the driver skeleton of
// grotz (mo_grotz.f90:119-176, :840-876).  The time loop itself is samsim_b200_step.  No physics here.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../../include/samsim_b200_host.h"

namespace {

const double rho_l = 1028.0, c_l = 3400.0;  // mo_parameters.f90:51,53
const double sigma_sb = 5.6704 * (double)1e-8f;  // mo_parameters.f90:59 (5.6704_wp*1e-8: the second factor is single precision)

void alloc_case(samsim_host_case_t* c) {
  const int N = c->cfg.Nlayer;
  for (int a = 0; a < SAMSIM_ARR_COUNT; a++) {
    int ext = N;
    if (a == SAMSIM_ARR_RAY) ext = N - 1;
    if (a == SAMSIM_ARR_FL_Q) ext = N + 1;
    c->arrays[a] = (double*)calloc((size_t)ext, sizeof(double));  // sub_allocate zero-fills, mo_init.f90:2082-2088
  }
}

void defaults(samsim_config_t* g) {  // mo_init.f90:83-109 and mo_parameters.f90:107-112
  memset(g, 0, sizeof *g);
  g->boundflux_flag = 1; g->atmoflux_flag = 1; g->albedo_flag = 2;
  g->grav_heat_flag = 1; g->flush_heat_flag = 1; g->flood_flag = 2; g->flush_flag = 5; g->grav_flag = 2; g->harmonic_flag = 2;
  g->prescribe_flag = 1; g->salt_flag = 1;
  g->turb_flag = 2; g->bottom_flag = 1; g->tank_flag = 1;
  g->precip_flag = 0; g->freeboard_snow_flag = 0; g->snow_flush_flag = 1; g->snow_precip_flag = 1;
  g->lab_snow_flag = 0;
  g->max_flux_plate = 10000.0; g->k_snow_flush = 0.75; g->k_styropor = 0.8;
}

// Fortran edit descriptors as the reference uses them (mo_output.f90:300-319): F9.3 / F9.5 / ES14.7 then 2x.
void put_F(FILE* f, double v, int w, int d) {
  char buf[64];
  int n = snprintf(buf, sizeof buf, "%*.*f", w, d, v);
  if (n > w) {  // Fortran prints w asterisks when the value does not fit
    for (int q = 0; q < w; q++) fputc('*', f);
  } else {
    fputs(buf, f);
  }
}
void put_ES(FILE* f, double v) {  // ES14.7
  char buf[64];
  snprintf(buf, sizeof buf, "%14.7E", v);
  fputs(buf, f);
}
void row_F(FILE* f, const double* a, int n, int w, int d) {
  for (int k = 0; k < n; k++) { put_F(f, a[k], w, d); fputs("  ", f); }
  fputc('\n', f);
}
void row_ES(FILE* f, const double* a, int n) {
  for (int k = 0; k < n; k++) { put_ES(f, a[k]); fputs("  ", f); }
  fputc('\n', f);
}

FILE* open_out(const std::string& dir, const char* name) { return fopen((dir + "/" + name).c_str(), "w"); }

// The dat_*.dat files of one run (output_begin / output_begin_bgc, mo_output.f90:276-339, :354-384) and the record
// output() writes at S8 (mo_output.f90:116-146, output_bgc :156-188).
struct OutFiles {
  FILE *T = nullptr, *psi_s = nullptr, *thick = nullptr, *S_bu = nullptr, *ray = nullptr, *psi_l = nullptr, *freeboard = nullptr,
       *snow = nullptr, *vital = nullptr, *grav = nullptr, *T2m = nullptr, *perm = nullptr, *flush_v = nullptr, *flush_h = nullptr,
       *psi_g = nullptr, *melt = nullptr;
  FILE* bgc[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  int N = 0, N_bgc = 0;

  std::vector<FILE**> all() {
    return {&T, &psi_s, &thick, &S_bu, &ray, &psi_l, &freeboard, &snow, &vital, &grav, &T2m, &perm, &flush_v, &flush_h, &psi_g, &melt,
            &bgc[0][0], &bgc[0][1], &bgc[1][0], &bgc[1][1]};
  }
  void close() {
    for (FILE** f : all())
      if (*f) { fclose(*f); *f = nullptr; }
  }
  // the 16 standard files must all open (the reference aborts in OPEN); then dat_settings.dat; then the tracer files
  int open(const std::string& out, const char* description, int32_t testcase, const samsim_host_case_t& cs, int32_t ncol) {
    const samsim_config_t& g = cs.cfg;
    N = g.Nlayer; N_bgc = g.N_bgc;
    T = open_out(out, "dat_T.dat"); psi_s = open_out(out, "dat_psi_s.dat"); thick = open_out(out, "dat_thick.dat");
    S_bu = open_out(out, "dat_S_bu.dat"); ray = open_out(out, "dat_ray.dat"); psi_l = open_out(out, "dat_psi_l.dat");
    freeboard = open_out(out, "dat_freeboard.dat"); snow = open_out(out, "dat_snow.dat");
    vital = open_out(out, "dat_vital_signs.dat"); grav = open_out(out, "dat_grav_drain.dat");
    T2m = open_out(out, "dat_T2m_T_top.dat"); perm = open_out(out, "dat_perm.dat"); flush_v = open_out(out, "dat_flush_v.dat");
    flush_h = open_out(out, "dat_flush_h.dat"); psi_g = open_out(out, "dat_psi_g.dat"); melt = open_out(out, "dat_melt.dat");
    for (FILE** f : all())
      if (f < &bgc[0][0] && !*f) return SAMSIM_ERR_STATE;
    FILE* s = open_out(out, "dat_settings.dat");
    if (s) {
      fprintf(s, " ################  Description  ###############\n %s\n #################  Testcase  #################\ntestcase         %8d\n", description ? description : "", testcase);
      fprintf(s, " ##############  Basic settings  ##############\ndt               %14.3f\nthick_0          %14.3f\ntime_out         %14.3f\ntime_total       %14.3f\n", g.dt, g.thick_0, g.time_out, cs.time_total);
      fprintf(s, "fl_q_bottom      %14.3f\nT_bottom         %14.3f\nS_bu_bottom      %14.3f\nN_top            %8d\nN_middle         %8d\nN_bottom         %8d\nNlayer           %8d\n",
              cs.scalars[SAMSIM_SC_FL_Q_BOTTOM], cs.scalars[SAMSIM_SC_T_BOTTOM], cs.scalars[SAMSIM_SC_S_BU_BOTTOM], g.N_top, g.N_middle, g.N_bottom, g.Nlayer);
      fprintf(s, " ##################  Flags  ###################\nboundflux_flag   %8d\natmoflux_flag    %8d\nalbedo_flag      %8d\ngrav_flag        %8d\nflush_flag       %8d\nflood_flag       %8d\ngrav_heat_flag   %8d\nflush_heat_flag  %8d\nharmonic_flag    %8d\nk_snow_flush     %14.3f\nprescribe_flag   %8d\nsalt_flag        %8d\nturb_flag        %8d\nbottom_flag      %8d\ntank_flag        %8d\nprecip_flag      %8d\n",
              g.boundflux_flag, g.atmoflux_flag, g.albedo_flag, g.grav_flag, g.flush_flag, g.flood_flag, g.grav_heat_flag, g.flush_heat_flag, g.harmonic_flag, g.k_snow_flush, g.prescribe_flag, g.salt_flag, g.turb_flag, g.bottom_flag, g.tank_flag, g.precip_flag);
      fprintf(s, " engine           %s\n ncol             %d\n", samsim_b200_version(), ncol);
      fclose(s);
    }
    for (int q = 0; q < N_bgc; q++) {  // dat_bgc0<k>.bu.dat / .br.dat per tracer
      char name[32];
      snprintf(name, sizeof name, "dat_bgc0%d.bu.dat", q + 1); bgc[q][0] = open_out(out, name);
      snprintf(name, sizeof name, "dat_bgc0%d.br.dat", q + 1); bgc[q][1] = open_out(out, name);
      if (!bgc[q][0] || !bgc[q][1]) return SAMSIM_ERR_STATE;
    }
    return SAMSIM_OK;
  }
  // one output record from a snapshot: ssc[SAMSIM_SNAPSC_COUNT], A[SAMSIM_SNAPARR_COUNT][N]
  void write(const double* ssc, const double* A) {
    row_F(T, A + (size_t)SAMSIM_SNAPARR_T * N, N, 9, 3);
    row_F(psi_s, A + (size_t)SAMSIM_SNAPARR_PSI_S * N, N, 9, 3);
    row_F(thick, A + (size_t)SAMSIM_SNAPARR_THICK * N, N, 9, 5);
    row_F(S_bu, A + (size_t)SAMSIM_SNAPARR_S_BU * N, N, 9, 3);
    row_F(ray, A + (size_t)SAMSIM_SNAPARR_RAY * N, N - 1, 9, 3);
    row_F(psi_l, A + (size_t)SAMSIM_SNAPARR_PSI_L * N, N, 9, 3);
    put_F(freeboard, ssc[SAMSIM_SNAPSC_FREEBOARD], 9, 3); fputc('\n', freeboard);
    put_F(snow, ssc[SAMSIM_SNAPSC_THICK_SNOW], 9, 3); fputs("  ", snow); put_F(snow, ssc[SAMSIM_SNAPSC_T_SNOW], 9, 3); fputs("  ", snow);
    put_F(snow, ssc[SAMSIM_SNAPSC_PSI_L_SNOW], 9, 3); fputs("  ", snow); put_F(snow, ssc[SAMSIM_SNAPSC_PSI_S_SNOW], 9, 3); fputc('\n', snow);
    put_F(vital, ssc[SAMSIM_SNAPSC_ENERGY_STORED], 15, 1);
    for (int q : {SAMSIM_SNAPSC_FRESHWATER, SAMSIM_SNAPSC_TOTAL_RESIST, SAMSIM_SNAPSC_THICKNESS, SAMSIM_SNAPSC_BULK_SALIN}) { fputs("  ", vital); put_F(vital, ssc[q], 10, 5); }
    fputc('\n', vital);
    put_F(grav, ssc[SAMSIM_SNAPSC_GRAV_DRAIN], 9, 6); fputs("  ", grav); put_F(grav, ssc[SAMSIM_SNAPSC_GRAV_SALT], 9, 5); fputs("  ", grav);
    put_F(grav, ssc[SAMSIM_SNAPSC_GRAV_TEMP], 7, 3); fputc('\n', grav);
    fprintf(T2m, "  %24.16E  %24.16E\n", ssc[SAMSIM_SNAPSC_T2M], ssc[SAMSIM_SNAPSC_T_TOP]);  // WRITE(45,*): list-directed, 17 digits
    row_ES(perm, A + (size_t)SAMSIM_SNAPARR_PERM * N, N);
    row_ES(flush_v, A + (size_t)SAMSIM_SNAPARR_FLUSH_V * N, N);
    row_ES(flush_h, A + (size_t)SAMSIM_SNAPARR_FLUSH_H * N, N);
    row_F(psi_g, A + (size_t)SAMSIM_SNAPARR_PSI_G * N, N, 9, 3);
    for (int q = 0; q < N_bgc; q++) {  // output_bgc, format_bgc = Nlayer x (F16.8,2x)
      if (bgc[q][0]) row_F(bgc[q][0], A + (size_t)(SAMSIM_SNAPARR_BGC1_BU + 2 * q) * N, N, 16, 8);
      if (bgc[q][1]) row_F(bgc[q][1], A + (size_t)(SAMSIM_SNAPARR_BGC1_BR + 2 * q) * N, N, 16, 8);
    }
    put_ES(melt, ssc[SAMSIM_SNAPSC_MELT_THICK_OUTPUT1]); fputs("  ", melt); put_ES(melt, ssc[SAMSIM_SNAPSC_MELT_THICK_OUTPUT2]); fputs("  ", melt);
    put_ES(melt, ssc[SAMSIM_SNAPSC_MELT_THICK_OUTPUT3]); fputc('\n', melt);
  }
};

// the initial column of one testcase into column `col` of the handle
int load_case(samsim_handle_t h, const samsim_host_case_t& cs, int32_t col) {
  int rc = 0;
  for (int a = 0; a < SAMSIM_ARR_COUNT && !rc; a++)
    if (samsim_b200_array_extent(h, a) > 0) rc = samsim_b200_set_array(h, a, cs.arrays[a], col, 1);
  for (int q = 0; q < SAMSIM_SC_COUNT && !rc; q++) rc = samsim_b200_set_scalar(h, q, &cs.scalars[q], col, 1);
  if (!rc) rc = samsim_b200_set_int(h, SAMSIM_INT_N_ACTIVE, &cs.N_active, col, 1);
  return rc;
}

// forcing of atmoflux_flag 2 (mo_grotz.f90:131-135): the four *.txt.input files, 13148 records
int set_reanalysis_forcing(samsim_handle_t h, const samsim_grotz_options_t* opt) {
  const int nrec = 13148;
  std::vector<double> series((size_t)4 * nrec);
  int rc = samsim_host_read_forcing(opt->forcing_dir, nrec, series.data());
  if (!rc) rc = samsim_b200_set_forcing(h, 1, nrec, series.data(), nullptr, opt->forcing_scale, opt->forcing_offset);
  return rc;
}

// The series a testcase reads in the prologue, in the kind order of samsim_b200_set_lab_forcing ([4][nrec]):
// 101-105 the four per-second lab series (mo_grotz.f90:138-169), length_input_lab records each; 8 Tinput.txt
// (mo_grotz.f90:138-143, one value per minute) and 111 Ts_<int(dt)>s.txt (mo_grotz.f90:171-176, one value per step)
// as Tice, as many records as the file holds.  nrec = 0: the testcase reads no series.
int read_case_series(const samsim_host_case_t& cs, int32_t testcase, const samsim_grotz_options_t* opt, std::vector<double>& lab,
                     int64_t& nrec) {
  nrec = 0;
  lab.clear();
  if (testcase == 8 || testcase == 111) {
    std::vector<double> T;
    char ts_name[64];
    snprintf(ts_name, sizeof ts_name, "/Ts_%ds.txt", (int)cs.cfg.dt);
    const std::string path = std::string(opt->lab_input_dir ? opt->lab_input_dir : "2017_input") + (testcase == 8 ? "/Tinput.txt" : ts_name);
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return SAMSIM_ERR_STATE;
    double x;
    while (fscanf(f, " %lf", &x) == 1) T.push_back(x);
    fclose(f);
    if (T.empty()) return SAMSIM_ERR_STATE;
    nrec = (int64_t)T.size();
    lab.assign(4 * T.size(), 0.0);
    for (size_t r = 0; r < T.size(); r++) lab[r] = T[r];
  } else if (testcase >= 101 && testcase <= 105) {
    nrec = cs.length_input_lab;
    lab.resize((size_t)4 * (size_t)nrec);
    return samsim_host_read_lab_series(opt->lab_input_dir, testcase, nrec, lab.data());
  }
  return SAMSIM_OK;
}

}  // namespace

extern "C" {

int samsim_host_init_testcase(int32_t testcase, samsim_host_case_t* c) {
  if (!c) return SAMSIM_ERR_ARG;
  memset(c, 0, sizeof *c);
  samsim_config_t* g = &c->cfg;
  defaults(g);
  g->testcase = testcase;
  double* sc = c->scalars;
  double T_top = 0.0, T_bottom = 0.0, S_bu_bottom = 0.0, fl_q_bottom = 0.0, time_out = 0.0, T2m = 0.0;
  int N_active = 1;
  const bool lab = (testcase >= 101 && testcase <= 105);
  if (testcase == 1) {  // mo_init.f90:865-945
    g->Nlayer = 90; g->N_top = 5; g->N_bottom = 5; g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    g->turb_flag = 1; g->boundflux_flag = 1; g->grav_heat_flag = 1; g->flush_flag = 1; g->salt_flag = 2;
    T_top = -5.0; T_bottom = -1.; S_bu_bottom = 34.; fl_q_bottom = 0.0;
    g->thick_0 = 0.002; g->dt = 1.0; time_out = 3600.0; c->time_total = time_out * 72.0;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    c->arrays[SAMSIM_ARR_M][0] = c->arrays[SAMSIM_ARR_THICK][0] * rho_l;
    c->arrays[SAMSIM_ARR_S_ABS][0] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][0];
    c->arrays[SAMSIM_ARR_H_ABS][0] = c->arrays[SAMSIM_ARR_M][0] * (T_bottom)*c_l;
  } else if (testcase == 8) {  // mo_init.f90:1451-1494 (field temperatures prescribe T_top; the series comes from Tinput.txt)
    g->Nlayer = 50; g->N_bottom = 5; g->N_top = 4; g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    g->boundflux_flag = 1; g->grav_flag = 2; g->flush_flag = 5; g->flood_flag = 2;
    T_top = -5.0; T_bottom = (double)(-1.8f); S_bu_bottom = 34.0; fl_q_bottom = 15.0;
    g->thick_0 = 0.005; g->dt = 1.0; time_out = 3600.0; c->time_total = time_out * 12.0 * 12.0;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    c->arrays[SAMSIM_ARR_M][0] = c->arrays[SAMSIM_ARR_THICK][0] * rho_l;
    c->arrays[SAMSIM_ARR_S_ABS][0] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][0];
    c->arrays[SAMSIM_ARR_H_ABS][0] = c->arrays[SAMSIM_ARR_M][0] * (T_bottom)*c_l;
  } else if (testcase == 111) {  // mo_init.f90:141-221 (the harp temperature series Ts_<dt>s.txt is read by samsim_grotz)
    g->Nlayer = 100; g->N_top = 10; g->N_bottom = 10; g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    c->length_input_lab = 860333;
    g->turb_flag = 1; g->boundflux_flag = 1; g->grav_heat_flag = 1; g->flush_flag = 1; g->salt_flag = 2;
    T_top = -2.0; T_bottom = -1.67; S_bu_bottom = 33.4079; fl_q_bottom = 0.;
    g->thick_0 = 0.01; g->dt = 3.0; time_out = 3600.0 * 2.0; c->time_total = 2580996.0;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    c->arrays[SAMSIM_ARR_M][0] = c->arrays[SAMSIM_ARR_THICK][0] * rho_l;
    c->arrays[SAMSIM_ARR_S_ABS][0] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][0];
    c->arrays[SAMSIM_ARR_H_ABS][0] = c->arrays[SAMSIM_ARR_M][0] * (T_bottom)*c_l;
  } else if (testcase == 4) {  // mo_init.f90:1127-1207
    g->Nlayer = 100; g->N_bottom = 20; g->N_top = 20; g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    g->atmoflux_flag = 2; g->precip_flag = 1; g->boundflux_flag = 2; g->snow_flush_flag = 1; g->flush_heat_flag = 2;
    g->snow_precip_flag = 1;
    T_bottom = -1.0; S_bu_bottom = 34.0;
    g->thick_0 = 0.01; time_out = 86400.0; c->time_total = time_out * 365.0 * 4.5; g->dt = 10.0;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    for (int k = 0; k < g->Nlayer; k++) {
      c->arrays[SAMSIM_ARR_M][k] = c->arrays[SAMSIM_ARR_THICK][k] * rho_l;
      c->arrays[SAMSIM_ARR_S_ABS][k] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][k];
      c->arrays[SAMSIM_ARR_H_ABS][k] = 0.0;
    }
  } else if (testcase == 2 || testcase == 6 || testcase == 9) {
    // cooling-chamber tanks: mo_init.f90:948-1042 (2), :1278-1357 (6), :1684-1776 (9)
    double tank_depth;
    if (testcase == 2) {
      fl_q_bottom = 10.0; g->alpha_flux_instable = 22.0; g->alpha_flux_stable = 15.0; tank_depth = 1.0;
      g->Nlayer = 100; g->N_bottom = 10; g->N_top = 3;
      T2m = -20.0; T_top = -18.0; T_bottom = 0.0; S_bu_bottom = 31.2;
      g->thick_0 = 0.01; time_out = 3600.0 * 6.0; c->time_total = time_out * 4.0 * 30.0; g->dt = 30.0;
    } else if (testcase == 6) {
      fl_q_bottom = 35.0; g->alpha_flux_instable = 22.0; g->alpha_flux_stable = 11.0; tank_depth = 0.159;
      g->Nlayer = 40; g->N_bottom = 3; g->N_top = 3;
      T2m = -18.0; T_top = -18.0; T_bottom = 0.0; S_bu_bottom = 31.2;
      g->thick_0 = 0.0025; time_out = 1800.0 / 2.0; c->time_total = time_out * 39.0 * 2.0 * 2.0; g->dt = 0.5;
    } else {
      fl_q_bottom = 10.0; g->alpha_flux_instable = 22.0; g->alpha_flux_stable = 15.0; tank_depth = 0.8;
      g->Nlayer = 100; g->N_bottom = 10; g->N_top = 3;
      T2m = -15.0; T_top = -10.0; T_bottom = -0.07; S_bu_bottom = 34.6;
      g->thick_0 = 0.005; time_out = 3600.0 * 2.0; c->time_total = time_out * 12.0 * 6.0; g->dt = 10.0;
    }
    g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    g->tank_flag = 2; g->boundflux_flag = 3; g->grav_heat_flag = 1;
    g->m_total = rho_l * tank_depth;
    sc[SAMSIM_SC_S_TOTAL] = rho_l * S_bu_bottom * tank_depth;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    for (int k = 0; k < g->Nlayer; k++) {
      c->arrays[SAMSIM_ARR_M][k] = c->arrays[SAMSIM_ARR_THICK][k] * rho_l;
      c->arrays[SAMSIM_ARR_S_ABS][k] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][k];
      c->arrays[SAMSIM_ARR_H_ABS][k] = c->arrays[SAMSIM_ARR_M][k] * T_bottom;
    }
  } else if (testcase == 33 || testcase == 34 || testcase == 99) {
    // three more chamber set-ups: mo_init.f90:1779-1873 (33, fresh water), :1876-1970 (34), :768-862 (99, snow on ice)
    const double tank_depth = 0.94;
    g->alpha_flux_instable = 22.0; g->alpha_flux_stable = 15.0;
    g->tank_flag = 2; g->boundflux_flag = 3; g->grav_heat_flag = 1;
    g->dt = 10.0;
    if (testcase == 99) {
      fl_q_bottom = 5.0;
      g->Nlayer = 20; g->N_bottom = 5; g->N_top = 5;
      g->precip_flag = 0; g->flush_flag = 1; g->flood_flag = 1; g->grav_flag = 2;
      T2m = -5.0; T_top = -2.0; T_bottom = -1.8; S_bu_bottom = 34.0;
      g->thick_0 = 0.05; time_out = 60.0 * 10.0; c->time_total = 3600.0 * 24.0 * 7.0;
    } else {
      fl_q_bottom = 10.0;
      g->Nlayer = 100; g->N_bottom = 10; g->N_top = 3;
      T2m = -15.0; T_top = -10.0; T_bottom = 0.5; S_bu_bottom = (testcase == 33) ? 0.13 : 34.9;
      g->thick_0 = 0.005;
      if (testcase == 33) { time_out = 60.0 * 5.0; c->time_total = time_out * 12.0 * 6.0; }
      else { time_out = 60.0 * 10.0; c->time_total = 86400.0 * 10.0; }
    }
    g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    g->m_total = rho_l * tank_depth;
    sc[SAMSIM_SC_S_TOTAL] = rho_l * S_bu_bottom * tank_depth;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    for (int k = 0; k < g->Nlayer; k++) {
      c->arrays[SAMSIM_ARR_M][k] = c->arrays[SAMSIM_ARR_THICK][k] * rho_l;
      c->arrays[SAMSIM_ARR_S_ABS][k] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][k];
      c->arrays[SAMSIM_ARR_H_ABS][k] = c->arrays[SAMSIM_ARR_M][k] * T_bottom;  // sic: no c_l
    }
  } else if (testcase == 50) {  // mo_init.f90:1497-1532: stable initial conditions for the convection studies
    g->Nlayer = 70; g->N_bottom = 5; g->N_top = 5; g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    g->boundflux_flag = 2;
    sc[SAMSIM_SC_FL_SW] = 0.0;
    sc[SAMSIM_SC_FL_REST] = sigma_sb * 4106877291.8310046;  // sigma*(zeroK-20._wp)**4._wp: a constant expression, folded with a correctly rounded power
    fl_q_bottom = 20.0; T_top = -20.0; T_bottom = -1.72; S_bu_bottom = 34.0;
    g->thick_0 = 0.005; time_out = 3600.0 * 24.0 * 30.0; g->dt = 10.0; c->time_total = time_out * 12.0 * 3.0;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    c->arrays[SAMSIM_ARR_M][0] = c->arrays[SAMSIM_ARR_THICK][0] * rho_l;
    c->arrays[SAMSIM_ARR_S_ABS][0] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][0];
    c->arrays[SAMSIM_ARR_H_ABS][0] = c->arrays[SAMSIM_ARR_M][0] * (T_bottom)*c_l;
  } else if (testcase == 3) {  // mo_init.f90:1045-1124
    g->Nlayer = 20; g->N_bottom = 5; g->N_top = 5; g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    g->atmoflux_flag = 1; g->precip_flag = 0; g->boundflux_flag = 2;
    fl_q_bottom = 8.0; T_bottom = -1.0; S_bu_bottom = 34.0;
    g->thick_0 = 0.03; time_out = 86400.0 * 3.5; c->time_total = time_out * 54.0 * 2.0 * 2.0; g->dt = 60.0;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    for (int k = 0; k < g->Nlayer; k++) {
      c->arrays[SAMSIM_ARR_M][k] = c->arrays[SAMSIM_ARR_THICK][k] * rho_l;
      c->arrays[SAMSIM_ARR_S_ABS][k] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][k];
      c->arrays[SAMSIM_ARR_H_ABS][k] = 0.0;
    }
  } else if (testcase == 5) {  // mo_init.f90:1210-1275
    g->Nlayer = 100; N_active = g->Nlayer; g->N_bottom = 10; g->N_top = 20; g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    g->boundflux_flag = 2; g->atmoflux_flag = 3; g->flush_heat_flag = 2;
    g->flush_flag = 5; g->grav_flag = 1; g->flood_flag = 1;
    sc[SAMSIM_SC_FL_SW] = 0.0;
    sc[SAMSIM_SC_FL_REST] = 7072810000.0 * sigma_sb;  // 290._wp**4*sigma
    fl_q_bottom = 15.0; S_bu_bottom = 5.0; T_bottom = 0.;
    g->thick_0 = 0.01; time_out = 3600.0 * 3.0; c->time_total = time_out * 24.0 * 10.0; g->dt = 10.0;
    alloc_case(c);
    for (int k = 0; k < g->Nlayer; k++) {
      c->arrays[SAMSIM_ARR_THICK][k] = g->thick_0;
      c->arrays[SAMSIM_ARR_M][k] = c->arrays[SAMSIM_ARR_THICK][k] * rho_l;
      c->arrays[SAMSIM_ARR_S_ABS][k] = c->arrays[SAMSIM_ARR_M][k] * S_bu_bottom;
      c->arrays[SAMSIM_ARR_H_ABS][k] = c->arrays[SAMSIM_ARR_M][k] * (-90.0) * c_l;
    }
  } else if (testcase == 7) {  // mo_init.f90:1360-1448
    g->Nlayer = 100; g->N_bottom = 20; g->N_top = 20; g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    g->atmoflux_flag = 2; g->precip_flag = 1; g->boundflux_flag = 2;
    g->albedo_flag = 1; g->grav_heat_flag = 2; g->flush_heat_flag = 2;
    g->flush_flag = 4; g->grav_flag = 3; g->flood_flag = 3;
    T_bottom = -1.0; S_bu_bottom = 34.0;
    g->thick_0 = 0.01; time_out = 86400.0 / 2.0; c->time_total = time_out * 365.0 * 9.0; g->dt = 10.0;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    for (int k = 0; k < g->Nlayer; k++) {
      c->arrays[SAMSIM_ARR_M][k] = c->arrays[SAMSIM_ARR_THICK][k] * rho_l;
      c->arrays[SAMSIM_ARR_S_ABS][k] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][k];
      c->arrays[SAMSIM_ARR_H_ABS][k] = 0.0;
    }
  } else if (lab) {  // mo_init.f90:222-767
    static const double Sb[5] = {25.6664555556, 26.1336777778, 26.0335888889, 27.0363, 31.5625333333};
    static const double tt[5] = {1625000.0, 1124000.0, 1283000.0, 2439000.0, 1549000.0};
    static const int64_t len[5] = {1628263, 1124187, 1283092, 2439729, 1549323};
    const int q = testcase - 101;
    const double tank_depth = 0.94;
    g->alpha_flux_instable = 22.0; g->alpha_flux_stable = 21.0;
    g->Nlayer = 200; g->N_bottom = 10; g->N_top = 5; g->N_middle = g->Nlayer - g->N_top - g->N_bottom;
    c->length_input_lab = len[q];
    g->tank_flag = 2; g->boundflux_flag = 3; g->precip_flag = 0; g->grav_heat_flag = 1; g->flush_flag = 5; g->flood_flag = 2;
    g->grav_flag = 2; g->lab_snow_flag = 1; g->freeboard_snow_flag = 1; g->snow_flush_flag = 1; g->flush_heat_flag = 2;
    g->snow_precip_flag = 1;
    T2m = 0.0; T_top = 0.0; T_bottom = -1.3; S_bu_bottom = Sb[q];
    g->thick_0 = 0.01; time_out = 60.0 * 60.0; c->time_total = tt[q]; g->dt = 1.0;
    g->m_total = rho_l * tank_depth;
    sc[SAMSIM_SC_S_TOTAL] = rho_l * S_bu_bottom * tank_depth;
    alloc_case(c);
    c->arrays[SAMSIM_ARR_THICK][0] = g->thick_0;
    for (int k = 0; k < g->Nlayer; k++) {
      c->arrays[SAMSIM_ARR_M][k] = c->arrays[SAMSIM_ARR_THICK][k] * rho_l;
      c->arrays[SAMSIM_ARR_S_ABS][k] = S_bu_bottom * c->arrays[SAMSIM_ARR_M][k];
      c->arrays[SAMSIM_ARR_H_ABS][k] = c->arrays[SAMSIM_ARR_M][k] * T_bottom;  // sic: no c_l (mo_init.f90:299)
    }
  } else {
    return SAMSIM_ERR_CONFIG;
  }
  // common tail, mo_init.f90:1982-2009
  for (int k = 0; k < g->Nlayer; k++) {
    c->arrays[SAMSIM_ARR_T][k] = T_bottom;
    c->arrays[SAMSIM_ARR_S_BU][k] = S_bu_bottom;
    c->arrays[SAMSIM_ARR_PSI_L][k] = 1.0;
  }
  g->thick_min = g->thick_0 / 2.0;
  g->time_out = time_out;
  c->i_time = (int32_t)(c->time_total / g->dt);
  g->i_time_out = (int32_t)(time_out / g->dt);
  c->N_active = N_active;
  sc[SAMSIM_SC_T_BOTTOM] = T_bottom; sc[SAMSIM_SC_T_TOP] = T_top; sc[SAMSIM_SC_S_BU_BOTTOM] = S_bu_bottom;
  sc[SAMSIM_SC_T2M] = T2m; sc[SAMSIM_SC_FL_Q_BOTTOM] = fl_q_bottom;
  {
    double sS = 0.0, sm = 0.0;  // bulk_salin = SUM(S_abs(1:N_active))/SUM(m(1:N_active)), mo_init.f90:2007
    for (int k = 0; k < N_active; k++) { sS = sS + c->arrays[SAMSIM_ARR_S_ABS][k]; sm = sm + c->arrays[SAMSIM_ARR_M][k]; }
    sc[SAMSIM_SC_BULK_SALIN] = sS / sm;
  }
  sc[SAMSIM_SC_TTOP_WARM] = -5.0; sc[SAMSIM_SC_TTOP_COLD] = -10.0; sc[SAMSIM_SC_OFLUX_AMP] = 7.0;
  // passive tracers (bgc_flag 2): testcase 1 (mo_init.f90:921-944), 2 (:1016-1040), 6 (:1331-1355)
  if (testcase == 1 || testcase == 2 || testcase == 6) {
    g->N_bgc = (testcase == 6) ? 1 : 2;
    const double tank_depth = (testcase == 2) ? 1.0 : 0.159;
    for (int q = 0; q < g->N_bgc; q++) {
      const double bottom = (testcase == 1) ? (q == 0 ? 400.0 : 500.0) : 385.0;
      sc[SAMSIM_SC_BGC_BOTTOM1 + q] = bottom;
      if (testcase != 1) sc[SAMSIM_SC_BGC_TOTAL1 + q] = bottom * rho_l * tank_depth;
      c->arrays[SAMSIM_ARR_BGC_ABS1 + q][0] = bottom * c->arrays[SAMSIM_ARR_M][0];
    }
  }
  return SAMSIM_OK;
}

void samsim_host_case_free(samsim_host_case_t* c) {
  if (!c) return;
  for (int a = 0; a < SAMSIM_ARR_COUNT; a++) { free(c->arrays[a]); c->arrays[a] = nullptr; }
}

int samsim_host_read_forcing(const char* dir, int32_t nrec, double* series) {
  static const char* names[4] = {"flux_sw.txt.input", "flux_lw.txt.input", "T2m.txt.input", "precip.txt.input"};
  if (!series || nrec < 1) return SAMSIM_ERR_ARG;
  const std::string d = dir ? dir : ".";
  for (int kind = 0; kind < 4; kind++) {
    FILE* f = fopen((d + "/" + names[kind]).c_str(), "r");
    if (!f) return SAMSIM_ERR_STATE;
    for (int r = 0; r < nrec; r++) {
      if (fscanf(f, "%lf", &series[(size_t)kind * nrec + r]) != 1) { fclose(f); return SAMSIM_ERR_STATE; }
    }
    fclose(f);
  }
  return SAMSIM_OK;
}

// lab series of testcases 101-105 (mo_grotz.f90:138-169): 2017_input/{Tice,snowfall,heat,styropor}_exp_<N>.txt with
// N = testcase - 100, list-directed reals, nrec = length_input_lab values each; series[kind*nrec + r] in the kind
// order of samsim_b200_set_lab_forcing.  (Tocean_exp_<N>.txt is read by the reference too but never used by the loop.)
int samsim_host_read_lab_series(const char* dir, int32_t testcase, int64_t nrec, double* series) {
  if (!series || nrec < 1 || testcase < 101 || testcase > 105) return SAMSIM_ERR_ARG;
  static const char* names[4] = {"Tice", "snowfall", "heat", "styropor"};
  const std::string d = dir ? dir : "2017_input";
  for (int kind = 0; kind < 4; kind++) {
    char file[64];
    snprintf(file, sizeof file, "%s_exp_%d.txt", names[kind], testcase - 100);
    FILE* f = fopen((d + "/" + file).c_str(), "r");
    if (!f) return SAMSIM_ERR_STATE;
    for (int64_t r = 0; r < nrec; r++) {
      if (fscanf(f, " %lf", &series[(size_t)kind * nrec + r]) != 1) { fclose(f); return SAMSIM_ERR_STATE; }
      int ch = fgetc(f);  // list-directed input accepts commas between values
      if (ch != ',' && ch != EOF) ungetc(ch, f);
    }
    fclose(f);
  }
  return SAMSIM_OK;
}

int samsim_grotz(int32_t testcase, const char* description, const samsim_grotz_options_t* opt) {
  if (!opt || opt->ncol < 1 || !opt->output_dir) return SAMSIM_ERR_ARG;
  samsim_host_case_t cs;
  int rc = samsim_host_init_testcase(testcase, &cs);
  if (rc) return rc;
  const samsim_config_t& g = cs.cfg;
  const int N = g.Nlayer;

  // ---- output_begin / output_settings (mo_output.f90:276-339, :41-106) ----
  OutFiles F;
  samsim_handle_t h = nullptr;
  auto finish = [&](int code) {  // every exit path: close the files, release the device and the host case
    F.close();
    if (h) samsim_b200_destroy(h);
    samsim_host_case_free(&cs);
    return code;
  };
  if ((rc = F.open(opt->output_dir, description, testcase, cs, opt->ncol))) return finish(rc);

  // ---- device ----
  rc = samsim_b200_create(&g, opt->ncol, opt->device, &h);
  if (rc) return finish(rc);
  rc = load_case(h, cs, 0);
  if (!rc) rc = samsim_b200_set_clock(h, 0.0, 0, 0, 1);
  if (!rc && opt->ncol > 1) rc = samsim_b200_broadcast_column(h, 0, 0, opt->ncol);
  if (!rc && opt->ttop_warm) rc = samsim_b200_set_scalar(h, SAMSIM_SC_TTOP_WARM, opt->ttop_warm, 0, opt->ncol);
  if (!rc && opt->ttop_warm) rc = samsim_b200_set_scalar(h, SAMSIM_SC_T_TOP, opt->ttop_warm, 0, opt->ncol);  // T_top starts at the warm level (mo_init.f90:894)
  if (!rc && opt->ttop_cold) rc = samsim_b200_set_scalar(h, SAMSIM_SC_TTOP_COLD, opt->ttop_cold, 0, opt->ncol);
  if (!rc && opt->oflux_amp) rc = samsim_b200_set_scalar(h, SAMSIM_SC_OFLUX_AMP, opt->oflux_amp, 0, opt->ncol);
  if (!rc && g.atmoflux_flag == 2) rc = set_reanalysis_forcing(h, opt);
  {
    std::vector<double> lab;
    int64_t nrec = 0;
    if (!rc) rc = read_case_series(cs, testcase, opt, lab, nrec);
    if (!rc && nrec > 0) rc = samsim_b200_set_lab_forcing(h, 1, nrec, lab.data(), nullptr);
  }
  if (!rc) rc = samsim_b200_set_snapshot_mode(h, SAMSIM_SNAP_FULL);

  // ---- the time loop in chunks that end on output steps (mo_grotz.f90:182, :340) ----
  const int64_t total = (opt->max_steps > 0 && opt->max_steps < cs.i_time) ? opt->max_steps : cs.i_time;
  int64_t done = 0;
  std::vector<double> ssc(SAMSIM_SNAPSC_COUNT), sar((size_t)SAMSIM_SNAPARR_COUNT * N);
  int32_t status = 0;
  while (!rc && done < total) {
    int64_t n = samsim_b200_steps_to_next_output(h);
    if (n <= 0) { rc = SAMSIM_ERR_STATE; break; }  // cannot happen with a consistent clock; never spin on step(h, 0)
    const bool wrote = (done + n <= total);
    if (n > total - done) n = total - done;
    rc = samsim_b200_step(h, n);
    if (rc) break;
    done += n;
    rc = samsim_b200_get_status(h, &status, 0, 1);
    if (rc || status) break;
    if (wrote) {  // S8: CALL output(...) (mo_output.f90:116-146) with the values the device captured there
      rc = samsim_b200_get_snapshot(h, ssc.data(), sar.data(), 0, 1);
      if (rc) break;
      F.write(ssc.data(), sar.data());
      if (!opt->quiet)
        printf("progress: %3d%%,  thickness: %6.3f m,  surface T: %7.3f C,  T2m: %7.3f\n", (int)(100.0 * ssc[SAMSIM_SNAPSC_TIME] / cs.time_total),
               ssc[SAMSIM_SNAPSC_THICKNESS], ssc[SAMSIM_SNAPSC_T_TOP], ssc[SAMSIM_SNAPSC_T2M]);
    }
  }
  return finish(rc ? rc : status);  // 0, a negative samsim_b200_err, or the reference STOP code of column 0
}

int samsim_grotz_batch(const samsim_grotz_member_t* m, int32_t n, const samsim_grotz_options_t* opt, int32_t* codes) {
  if (!m || n < 1 || !opt || !codes) return SAMSIM_ERR_ARG;
  if (opt->ncol != 0 || opt->output_dir || opt->max_steps != 0 || opt->forcing_scale || opt->forcing_offset || opt->ttop_warm ||
      opt->ttop_cold || opt->oflux_amp)
    return SAMSIM_ERR_ARG;  // these belong to a member or to samsim_grotz's identical columns
  for (int32_t q = 0; q < n; q++)
    if (!m[q].output_dir || m[q].max_steps < 0) return SAMSIM_ERR_ARG;
  std::vector<samsim_host_case_t> cs((size_t)n);
  std::vector<OutFiles> F((size_t)n);
  int32_t ninit = 0;
  samsim_handle_t h = nullptr;
  auto finish = [&](int code) {  // every exit path: close the files, release the device and the host cases
    for (OutFiles& f : F) f.close();
    if (h) samsim_b200_destroy(h);
    for (int32_t q = 0; q < ninit; q++) samsim_host_case_free(&cs[q]);
    return code;
  };
  // ---- init(testcase) of every member; one run-wide configuration, checked before any device call ----
  int rc = 0;
  for (; ninit < n; ninit++)
    if ((rc = samsim_host_init_testcase(m[ninit].testcase, &cs[ninit]))) return finish(rc);
  const samsim_config_t& g = cs[0].cfg;
  auto lab = [](int32_t tc) { return tc >= 101 && tc <= 105; };
  for (int32_t q = 1; q < n; q++) {
    samsim_config_t c = cs[q].cfg;
    if (lab(c.testcase) && lab(g.testcase)) c.testcase = g.testcase;  // the five lab experiments take one device path
    if (memcmp(&c, &g, sizeof c) != 0) return finish(SAMSIM_ERR_CONFIG);
  }
  const int N = g.Nlayer;
  for (int32_t q = 0; q < n && !rc; q++) rc = F[q].open(m[q].output_dir, m[q].description, m[q].testcase, cs[q], n);
  if (rc) return finish(rc);

  // ---- device: member q is column q and reads lab set q ----
  if ((rc = samsim_b200_create(&g, n, opt->device, &h))) return finish(rc);
  for (int32_t q = 0; q < n && !rc; q++) rc = load_case(h, cs[q], q);
  if (!rc) rc = samsim_b200_set_clock(h, 0.0, 0, 0, 1);
  if (!rc && g.atmoflux_flag == 2) rc = set_reanalysis_forcing(h, opt);
  {
    std::vector<std::vector<double>> series((size_t)n);
    std::vector<int64_t> len((size_t)n, 0);
    int64_t nrec = 0;
    for (int32_t q = 0; q < n && !rc; q++) {
      rc = read_case_series(cs[q], m[q].testcase, opt, series[q], len[q]);
      nrec = std::max(nrec, len[q]);
    }
    if (!rc && nrec > 0) {  // one table padded to the longest series; each set keeps its own length
      std::vector<double> table((size_t)n * 4 * (size_t)nrec, 0.0);
      std::vector<int32_t> set_of_col((size_t)n);
      for (int32_t q = 0; q < n; q++) {
        set_of_col[q] = q;
        for (int kind = 0; kind < 4; kind++)
          std::copy(series[q].begin() + (size_t)kind * len[q], series[q].begin() + (size_t)(kind + 1) * len[q],
                    table.begin() + ((size_t)q * 4 + kind) * (size_t)nrec);
      }
      rc = samsim_b200_set_lab_forcing(h, n, nrec, table.data(), set_of_col.data());
      if (!rc) rc = samsim_b200_set_lab_lengths(h, n, len.data());
    }
  }
  std::vector<int64_t> end((size_t)n);
  int64_t total = 0;
  for (int32_t q = 0; q < n; q++) {
    end[q] = (m[q].max_steps > 0 && m[q].max_steps < cs[q].i_time) ? m[q].max_steps : cs[q].i_time;
    total = std::max(total, end[q]);
  }
  if (!rc) rc = samsim_b200_set_end_step(h, end.data(), 0, n);
  if (!rc) rc = samsim_b200_set_snapshot_mode(h, SAMSIM_SNAP_FULL);

  // ---- the time loop of samsim_grotz up to the latest end; a member writes while it runs and its status is 0 ----
  int64_t done = 0;
  std::vector<double> ssc((size_t)n * SAMSIM_SNAPSC_COUNT), sar((size_t)n * SAMSIM_SNAPARR_COUNT * N);
  std::vector<int32_t> status((size_t)n, 0);
  while (!rc && done < total) {
    int64_t k = samsim_b200_steps_to_next_output(h);
    if (k <= 0) { rc = SAMSIM_ERR_STATE; break; }
    const bool wrote = (done + k <= total);
    if (k > total - done) k = total - done;
    if ((rc = samsim_b200_step(h, k))) break;
    done += k;
    if ((rc = samsim_b200_get_status(h, status.data(), 0, n))) break;
    bool running = false;
    for (int32_t q = 0; q < n; q++) running = running || (status[q] == 0 && done < end[q]);
    if (wrote) {
      if ((rc = samsim_b200_get_snapshot(h, ssc.data(), sar.data(), 0, n))) break;
      for (int32_t q = 0; q < n; q++) {
        if (status[q] != 0 || done > end[q]) continue;
        const double* sc = ssc.data() + (size_t)q * SAMSIM_SNAPSC_COUNT;
        F[q].write(sc, sar.data() + (size_t)q * SAMSIM_SNAPARR_COUNT * N);
        if (!opt->quiet)
          printf("member %d progress: %3d%%,  thickness: %6.3f m,  surface T: %7.3f C,  T2m: %7.3f\n", q,
                 (int)(100.0 * sc[SAMSIM_SNAPSC_TIME] / cs[q].time_total), sc[SAMSIM_SNAPSC_THICKNESS], sc[SAMSIM_SNAPSC_T_TOP],
                 sc[SAMSIM_SNAPSC_T2M]);
      }
    }
    if (!running) break;  // every member has failed or reached its end
  }
  for (int32_t q = 0; q < n; q++) codes[q] = rc ? rc : status[q];
  return finish(rc);
}

}  // extern "C"
