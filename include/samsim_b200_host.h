/* samsim_b200_host.h -- C++ host side above the C ABI: the batched mirror of the reference's entry point
 *     SUBROUTINE grotz(testcase, description)          mo_grotz.f90:83
 * for environments without a Fortran compiler (this image).  It does what the Fortran prologue/epilogue do --
 * init(testcase) (mo_init.f90:73; testcases 1, 4, 101-105), sub_input (mo_functions.f90:304-327),
 * output_begin/output_settings/output (mo_output.f90:41-146, 276-339) -- and drives the device through
 * include/samsim_b200.h.  With a Fortran toolchain, fortran/mo_grotz_b200.f90 is the drop-in instead.
 */
#ifndef SAMSIM_B200_HOST_H
#define SAMSIM_B200_HOST_H
#include <stdint.h>
#include "samsim_b200.h"
#ifdef __cplusplus
extern "C" {
#endif

/* one column of mo_data after init(testcase): arrays of extent Nlayer (fl_Q: Nlayer+1, ray: Nlayer-1), owned by the struct */
typedef struct {
  samsim_config_t cfg;
  int32_t N_active, i_time;            /* i_time = INT(time_total/dt), mo_init.f90:1998 */
  double time_total;
  double* arrays[SAMSIM_ARR_COUNT];
  double scalars[SAMSIM_SC_COUNT];
  int64_t length_input_lab;            /* testcases 101-105 */
} samsim_host_case_t;

/* mo_init.f90: defaults :83-132, testcase 1 :865-945, 2 :948-1042, 3 :1045-1124, 4 :1127-1207, 5 :1210-1275,
 * 6 :1278-1357, 7 :1360-1448, 9 :1684-1776, 33 :1779-1873, 34 :1876-1970, 50 :1497-1532, 99 :768-862, 101-105 :222-767,
 * 111 :141-221 (its series <lab_input_dir>/Ts_<int(dt)>s.txt is read by samsim_grotz, mo_grotz.f90:171-176), tail :1982-2009.
 * 8 :1451-1494 (its field temperature series input/DNotz_fieldT/Tinput.txt is read by samsim_grotz).
 * Returns SAMSIM_ERR_CONFIG for other testcases (the reference STOPs with 4321 for unknown ones; 51 is a table of 280
 * restart values: not covered). */
int samsim_host_init_testcase(int32_t testcase, samsim_host_case_t* out);
void samsim_host_case_free(samsim_host_case_t* c);

/* sub_input (mo_functions.f90:304-327): first nrec values of flux_sw/flux_lw/T2m/precip.txt.input in `dir`,
 * series[kind*nrec + r] in samsim_forcing_kind order. */
int samsim_host_read_forcing(const char* dir, int32_t nrec, double* series);

/* mo_grotz.f90:138-169: the per-second lab series of testcases 101-105, nrec = length_input_lab values per file;
 * series[kind*nrec + r], kinds 0 Tice, 1 snowfall, 2 heat, 3 styropor (the order of samsim_b200_set_lab_forcing). */
int samsim_host_read_lab_series(const char* dir, int32_t testcase, int64_t nrec, double* series);

typedef struct {
  int32_t ncol;              /* >= 1; column 0 writes the output files */
  int32_t device;
  const char* forcing_dir;   /* directory with the four *.txt.input files (atmoflux_flag 2); NULL = "." */
  const char* output_dir;    /* directory for dat_*.dat; must exist (the reference needs ./output) */
  int64_t max_steps;         /* 0 = i_time */
  /* optional per-column perturbations (NULL = identical columns): forcing scale/offset [4][ncol], and scalars */
  const double* forcing_scale;
  const double* forcing_offset;
  const double* ttop_warm; const double* ttop_cold; const double* oflux_amp;   /* [ncol] each or NULL */
  int32_t quiet;
  const char* lab_input_dir; /* testcases 101-105: directory with {Tice,snowfall,heat,styropor}_exp_<N>.txt
                                (mo_grotz.f90:138-169); NULL = "2017_input" like the reference */
} samsim_grotz_options_t;

/* grotz(testcase, description) for ncol columns: init, forcing, time loop on the device, dat_*.dat in the reference's
 * formats for column 0.  Returns 0, a negative samsim_b200_err, or the positive reference STOP code of column 0. */
int samsim_grotz(int32_t testcase, const char* description, const samsim_grotz_options_t* opt);

/* one member of samsim_grotz_batch: a testcase run of its own length with its own dat_*.dat files */
typedef struct {
  int32_t testcase;
  const char* description;
  const char* output_dir;    /* must exist */
  int64_t max_steps;         /* 0 = i_time of the testcase */
} samsim_grotz_member_t;

/* grotz(testcase, description) for n members at once, one column each, e.g. the five lab experiments 101-105 of
 * different durations.  Every member's testcase must give the same samsim_config_t, except that testcases 101-105
 * may be mixed (else SAMSIM_ERR_CONFIG, before any device call).  opt supplies device, forcing_dir, lab_input_dir and
 * quiet; its ncol, output_dir, max_steps and perturbation pointers must be 0 / NULL (else SAMSIM_ERR_ARG).  Member q
 * reads its own series (101-105: length_input_lab records) and runs min(i_time, max_steps) steps; it writes the
 * records samsim_grotz(testcase, description) with that max_steps writes, byte for byte except the ncol line of
 * dat_settings.dat, and stops writing when its status turns non-zero while the others go on.  codes[q] = 0, a
 * negative samsim_b200_err or the member's STOP code.  Returns 0 or a negative samsim_b200_err. */
int samsim_grotz_batch(const samsim_grotz_member_t* m, int32_t n, const samsim_grotz_options_t* opt, int32_t* codes);

#ifdef __cplusplus
}
#endif
#endif
