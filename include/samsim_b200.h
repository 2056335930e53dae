/* samsim_b200.h -- C ABI of the B200 column-timestep engine.
 *
 * Drop-in boundary.  The reference has no FFI; its seam is the Fortran entry
 *     SUBROUTINE grotz(testcase, description)            mo_grotz.f90:83
 * and the module-global state of mo_data (mo_data.f90:34-203).  Inside grotz the
 * replaceable unit is the body of `DO i = 1,i_time` (mo_grotz.f90:182-835).  The functions
 * below are what an ISO_C_BINDING shim (fortran/mo_samsim_b200.f90, see INTEGRATION.md)
 * binds to replace that loop body for a BATCH of independent columns:
 *
 *   reference (one column, host)                         this library (ncol columns, device)
 *   ---------------------------------------------------  ------------------------------------
 *   init(testcase) fills mo_data   mo_init.f90:73        samsim_b200_create + _set_array/_set_scalar
 *   sub_input reads 4 series       mo_functions.f90:304  samsim_b200_set_forcing (+ per-column affine)
 *   lab series READs               mo_grotz.f90:138-169  samsim_b200_set_lab_forcing
 *   DO i = 1,i_time ... END DO     mo_grotz.f90:182-835  samsim_b200_step(h, nsteps)
 *   CALL output(...) at S8         mo_grotz.f90:340-398  samsim_b200_get_snapshot (values captured at S8)
 *   STOP <code>                    SURVEY section 4      per-column status, samsim_b200_get_status
 *   mo_data arrays after the loop                        samsim_b200_get_array/_get_scalar
 *
 * Conventions: every function returns 0 on success or a negative samsim_b200_err; no
 * exceptions or exit() cross the ABI.  All reals are IEEE double (REAL(wp),
 * mo_parameters.f90:33), all integers int32 (default INTEGER).  Host arrays are
 * column-major per column, i.e. host[c*extent + (k-1)] is Fortran element k of column c --
 * for ncol = 1 that is exactly the Fortran ALLOCATABLE.  Device memory is owned by the
 * library.  One host thread per handle; one handle per device.
 */
#ifndef SAMSIM_B200_H
#define SAMSIM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct samsim_b200_handle_s* samsim_handle_t;

typedef enum {
  SAMSIM_OK = 0,
  SAMSIM_ERR_ARG = -1,       /* bad argument (null pointer, range, unknown id) */
  SAMSIM_ERR_CUDA = -2,      /* CUDA runtime error; text via samsim_b200_last_error */
  SAMSIM_ERR_NO_DEVICE = -3, /* no CUDA device: there is NO CPU fallback */
  SAMSIM_ERR_CONFIG = -4,    /* configuration not accepted (inconsistent grid, unknown flag value, N_bgc > 2) */
  SAMSIM_ERR_STATE = -5      /* call order (forcing missing, snapshot disabled, ...) */
} samsim_b200_err;

/* Run-wide configuration = the flags of mo_data.f90:136-155 + grid/timestep scalars of
 * mo_data.f90:57-74 + the three mutable parameters of mo_parameters.f90:107-112.
 * Everything here is uniform over the batch. */
typedef struct {
  int32_t testcase;      /* selects the S15 hook (mo_grotz.f90:503-563): 1 sub_test1, 4|7 sub_test4, 101..105 lab tables, else none */
  int32_t Nlayer, N_top, N_middle, N_bottom;
  int32_t atmoflux_flag, grav_flag, prescribe_flag, grav_heat_flag, flush_heat_flag, turb_flag, salt_flag,
      boundflux_flag, flush_flag, flood_flag, bottom_flag, precip_flag, harmonic_flag, tank_flag, albedo_flag,
      lab_snow_flag, freeboard_snow_flag, snow_flush_flag, snow_precip_flag;
  int32_t i_time_out;    /* INT(time_out/dt), mo_init.f90:1999: a record every i_time_out+1 steps */
  int32_t N_bgc;         /* passive tracers: 0 = bgc_flag 1 (none); 1 or 2 = bgc_flag 2 with N_bgc tracers (mo_data.f90 bgc_*) */
  double dt, thick_0, thick_min, time_out;
  double alpha_flux_instable, alpha_flux_stable; /* mo_data.f90:132-133 */
  double m_total;        /* tank_flag 2 (mo_data.f90:195); S_total is per column (SAMSIM_SC_S_TOTAL) */
  double max_flux_plate, k_snow_flush, k_styropor; /* mo_parameters.f90:107-112 */
} samsim_config_t;

/* Per-layer arrays of mo_data (extent Nlayer unless noted).  Arrays that are dead at a step
 * boundary in the reference (H, S_br, V_ex, fl_m, fl_rad, flush_*_old: always rewritten before
 * they are read) are not part of the device state. */
typedef enum {
  SAMSIM_ARR_M = 0,     /* m      mo_data.f90:44 */
  SAMSIM_ARR_S_ABS,     /* S_abs  :41 */
  SAMSIM_ARR_H_ABS,     /* H_abs  :35 */
  SAMSIM_ARR_THICK,     /* thick  :43 */
  SAMSIM_ARR_T,         /* T      :38 */
  SAMSIM_ARR_PHI,       /* phi    :50 */
  SAMSIM_ARR_S_BU,      /* S_bu   :39 */
  SAMSIM_ARR_PSI_S,     /* psi_s  :51 */
  SAMSIM_ARR_PSI_L,     /* psi_l  :52 */
  SAMSIM_ARR_PSI_G,     /* psi_g  :53 */
  SAMSIM_ARR_RAY,       /* ray    :54, extent Nlayer-1 */
  SAMSIM_ARR_PERM,      /* perm   :55 */
  SAMSIM_ARR_FLUSH_V,   /* flush_v :55 */
  SAMSIM_ARR_FLUSH_H,   /* flush_h :55 */
  SAMSIM_ARR_FL_Q,      /* fl_Q   :37, extent Nlayer+1 */
  SAMSIM_ARR_BGC_ABS1,  /* bgc_abs(:,1), only with N_bgc >= 1 (array_extent returns -1 otherwise) */
  SAMSIM_ARR_BGC_ABS2,  /* bgc_abs(:,2), only with N_bgc == 2 */
  SAMSIM_ARR_COUNT
} samsim_array_id;

/* Per-column double scalars of mo_data (Appendix D of SURVEY.md) + the per-column knobs. */
typedef enum {
  SAMSIM_SC_T_BOTTOM = 0, SAMSIM_SC_T_TOP, SAMSIM_SC_S_BU_BOTTOM, SAMSIM_SC_T2M, SAMSIM_SC_FL_Q_BOTTOM, /* mo_data.f90:80-84 */
  SAMSIM_SC_PSI_S_SNOW, SAMSIM_SC_PSI_L_SNOW, SAMSIM_SC_PSI_G_SNOW, SAMSIM_SC_PHI_S, SAMSIM_SC_S_ABS_SNOW,
  SAMSIM_SC_H_ABS_SNOW, SAMSIM_SC_M_SNOW, SAMSIM_SC_T_SNOW, SAMSIM_SC_THICK_SNOW, SAMSIM_SC_LIQUID_PRECIP,
  SAMSIM_SC_SOLID_PRECIP, SAMSIM_SC_FL_Q_SNOW,                                                           /* :87-98 */
  SAMSIM_SC_ENERGY_STORED, SAMSIM_SC_TOTAL_RESIST, SAMSIM_SC_FRESHWATER, SAMSIM_SC_THICKNESS, SAMSIM_SC_BULK_SALIN, /* :101-106 */
  SAMSIM_SC_ALBEDO, SAMSIM_SC_FL_SW, SAMSIM_SC_FL_LW, SAMSIM_SC_FL_REST,                                 /* :113-118 */
  SAMSIM_SC_GRAV_DRAIN, SAMSIM_SC_GRAV_SALT, SAMSIM_SC_GRAV_TEMP,                                        /* :122-124 */
  SAMSIM_SC_MELT_THICK, SAMSIM_SC_MELT_THICK_SNOW, SAMSIM_SC_MELT_THICK_SNOW_OLD,                         /* :127-128 */
  SAMSIM_SC_MELT_THICK_OUTPUT1, SAMSIM_SC_MELT_THICK_OUTPUT2, SAMSIM_SC_MELT_THICK_OUTPUT3,               /* :129 */
  SAMSIM_SC_FREEBOARD, SAMSIM_SC_T_FREEZE, SAMSIM_SC_MELT_ERR, SAMSIM_SC_S_TOTAL,                         /* :60-61, :202, :196 */
  /* literals of the reference promoted to per-column knobs; the identity values reproduce the reference */
  SAMSIM_SC_TTOP_WARM,  /* -5  in sub_test1, mo_testcase_specifics.f90:46-87 */
  SAMSIM_SC_TTOP_COLD,  /* -10 in sub_test1 */
  SAMSIM_SC_OFLUX_AMP,  /* 7 W/m2 in sub_test4, mo_testcase_specifics.f90:200 */
  SAMSIM_SC_BGC_BOTTOM1, SAMSIM_SC_BGC_BOTTOM2, /* bgc_bottom(1:2): tracer concentration of the water below */
  SAMSIM_SC_BGC_TOTAL1, SAMSIM_SC_BGC_TOTAL2,   /* bgc_total(1:2): tank budget (tank_flag 2) */
  SAMSIM_SC_COUNT
} samsim_scalar_id;

typedef enum {
  SAMSIM_INT_N_ACTIVE = 0, /* mo_data.f90:66 */
  SAMSIM_INT_STATUS,       /* 0 or the reference's STOP code (99, 98, 16, 345, 9876, 21234, 1337, 431, 7889) */
  SAMSIM_INT_STYROPOR_FLAG,/* :69 */
  SAMSIM_INT_EVENTS0,      /* branch events 0..31 (samsim_event_id): bit set once the column has executed the branch */
  SAMSIM_INT_EVENTS1,      /* branch events 32..63 */
  SAMSIM_INT_COUNT
} samsim_int_id;

/* Branch events.  Not in the reference (it has one column and PRINTs under debug_flag 2, e.g.
 * mo_layer_dynamics.f90:78-80): a per-column bit mask that records which rarely taken branches of the path a column
 * has executed since the words were last cleared (samsim_b200_set_int with zeros).  Bit id of
 * SAMSIM_INT_EVENTS0 (id < 32) / SAMSIM_INT_EVENTS1 (id - 32).  The parity tests assert these next to the CPU
 * oracle's counters of the same branches, so a test that claims to cover a branch proves that it ran. */
typedef enum {
  SAMSIM_EV_FLOOD = 0,            /* flood                          mo_flood.f90:55 */
  SAMSIM_EV_FLOOD_NEG_FREE,       /*   instant flooding beyond neg_free          :117-138 */
  SAMSIM_EV_FLOOD_SIMPLE,         /* flood_simple                   mo_flood.f90:167 */
  SAMSIM_EV_FLUSH3,               /* flush3                         mo_flush.f90:70 */
  SAMSIM_EV_FLUSH4,               /* flush4                         mo_flush.f90:253 */
  SAMSIM_EV_FLUSH_INLINE,         /* flush_flag 4                   mo_grotz.f90:704-713 */
  SAMSIM_EV_STYROPOR,             /* sub_fl_Q_styropor              mo_thermo_functions.f90:276 (call: mo_heat_fluxes.f90:202-258) */
  SAMSIM_EV_SNOW_THERMO,          /* snow_thermo (snow_flush_flag 0) mo_snow.f90:212 */
  SAMSIM_EV_SNOW_THERMO_MELTWATER,/* snow_thermo_meltwater          mo_snow.f90:331 */
  SAMSIM_EV_SNOW_WET,             /*   saturated-layer branch       :271 / :398 */
  SAMSIM_EV_SNOW_MERGE,           /*   snow without gas joins layer 1 :296 / :431 */
  SAMSIM_EV_SNOW_COMPACTION,      /*   psi_s_old > psi_s_snow       :253-263 */
  SAMSIM_EV_SNOW_COUPLING_ITER,   /* snow_coupling, iterative branch mo_snow.f90:87-98 */
  SAMSIM_EV_SNOW_COUPLING_WARM1,  /*   :76-80 */
  SAMSIM_EV_SNOW_COUPLING_WARM2,  /*   :81-85 */
  SAMSIM_EV_SNOW_PRECIP,          /* snow_precip                    mo_snow.f90:123 */
  SAMSIM_EV_SNOW_PRECIP_0,        /* snow_precip_0                  mo_snow.f90:167 */
  SAMSIM_EV_MELT_SNOW_ALL,        /* sub_melt_snow, all snow floods mo_functions.f90:453 */
  SAMSIM_EV_MELT_SNOW_PART,       /*   partial                      :461 */
  SAMSIM_EV_BOTTOM_MELT,          /* bottom_melt                    mo_layer_dynamics.f90:85 -> :341 */
  SAMSIM_EV_BOTTOM_MELT_SIMPLE_A, /* bottom_melt_simple, N_active < Nlayer   :95 */
  SAMSIM_EV_BOTTOM_MELT_SIMPLE_B, /* bottom_melt_simple, grid full, middle = thick_0   :106 */
  SAMSIM_EV_BOTTOM_GROWTH_SIMPLE, /* bottom_growth_simple           :122 -> :537 */
  SAMSIM_EV_BOTTOM_GROWTH,        /* bottom_growth                  :132 -> :438 */
  SAMSIM_EV_TOP_GROW_A,           /* top_grow, N_active <= N_top    :656 */
  SAMSIM_EV_TOP_GROW_B,           /* top_grow, N_top < N_active < Nlayer   :665 */
  SAMSIM_EV_TOP_GROW_C,           /* top_grow, N_active == Nlayer   :679 */
  SAMSIM_EV_TOP_MELT_A,           /* top_melt, N_active <= N_top    :244 */
  SAMSIM_EV_TOP_MELT_B,           /* top_melt, middle layers at thick_0   :253 */
  SAMSIM_EV_TOP_MELT_C,           /* top_melt, middle layers shrink :272 */
  SAMSIM_EV_GRAV_DRAINED,         /* fl_grav_drain: a layer above ray_crit drained   mo_grav_drain.f90:145 */
  SAMSIM_EV_SALT_CLAMP,           /* negative S_abs clamped         mo_grotz.f90:812-818 */
  SAMSIM_EV_GAS_REFILL,           /* gas in the lowest layer replaced by ocean water   mo_grotz.f90:405-410 */
  SAMSIM_EV_GETT_TFR_FALLBACK,    /* getT: iterate outside [-200, 0] restarts at T_fr   mo_thermo_functions.f90:101 */
  SAMSIM_EV_GETT_SALTFREE,        /* getT: salt-free branch         :127-137 */
  SAMSIM_EV_GETT_LIQUID,          /* getT: liquid layer             :138-140 */
  SAMSIM_EV_HEAT_MELT,            /* sub_heat_fluxes: surface at the melting point   mo_heat_fluxes.f90:167-180 */
  SAMSIM_EV_HEAT_THIN_SNOW,       /* sub_heat_fluxes: thin snow coupled to layer 1   :291-295 */
  SAMSIM_EV_MELT_THICK_GAS,       /* sub_melt_thick: gas-fraction correction   mo_functions.f90:418-426 */
  SAMSIM_EV_SNOW_MELTWATER_TO_ICE,/* snow melt water added to layer 1   mo_grotz.f90:677-685 */
  SAMSIM_EV_PRESCRIBE,            /* prescribe_flag 2               mo_grotz.f90:482-497 */
  SAMSIM_EV_GRAV_DRAIN_SIMPLE,    /* fl_grav_drain_simple           mo_grav_drain.f90:218 */
  SAMSIM_EV_NOTZFLUX,             /* sub_notzflux                   mo_functions.f90:270 */
  SAMSIM_EV_FLUSH3_CLAMP,         /* flush3: negative S_abs clamped mo_flush.f90:218-227 */
  SAMSIM_EV_SCRUB,                /* layer below N_active scrubbed  mo_grotz.f90:772-783 */
  SAMSIM_EV_MELT_THICK,           /* sub_melt_thick called          mo_functions.f90:386 */
  SAMSIM_EV_TURB,                 /* sub_turb_flux                  mo_functions.f90:347 */
  SAMSIM_EV_TANK,                 /* tank salinity                  mo_grotz.f90:573-578 */
  SAMSIM_EV_TWO_PASS_STEP,        /* (device only) the column took the merged forward / backward passes of step.cuh in some step */
  SAMSIM_EV_COUNT
} samsim_event_id;

/* forcing kinds for samsim_b200_set_forcing, in sub_input's order of use */
typedef enum { SAMSIM_F_FL_SW = 0, SAMSIM_F_FL_LW = 1, SAMSIM_F_T2M = 2, SAMSIM_F_PRECIP = 3, SAMSIM_F_COUNT = 4 } samsim_forcing_kind;

/* what S8 captures for the host (mo_output.f90:116-146) */
typedef enum { SAMSIM_SNAP_NONE = 0, SAMSIM_SNAP_SCALARS = 1, SAMSIM_SNAP_FULL = 2 } samsim_snapshot_mode;
typedef enum {
  SAMSIM_SNAPSC_FREEBOARD = 0, SAMSIM_SNAPSC_THICK_SNOW, SAMSIM_SNAPSC_T_SNOW, SAMSIM_SNAPSC_PSI_L_SNOW,
  SAMSIM_SNAPSC_PSI_S_SNOW, SAMSIM_SNAPSC_ENERGY_STORED, SAMSIM_SNAPSC_FRESHWATER, SAMSIM_SNAPSC_TOTAL_RESIST,
  SAMSIM_SNAPSC_THICKNESS, SAMSIM_SNAPSC_BULK_SALIN, SAMSIM_SNAPSC_GRAV_DRAIN, SAMSIM_SNAPSC_GRAV_SALT,
  SAMSIM_SNAPSC_GRAV_TEMP, SAMSIM_SNAPSC_T2M, SAMSIM_SNAPSC_T_TOP, SAMSIM_SNAPSC_MELT_THICK_OUTPUT1,
  SAMSIM_SNAPSC_MELT_THICK_OUTPUT2, SAMSIM_SNAPSC_MELT_THICK_OUTPUT3, SAMSIM_SNAPSC_TIME, SAMSIM_SNAPSC_N_ACTIVE,
  SAMSIM_SNAPSC_COUNT
} samsim_snapshot_scalar_id;
/* arrays in a full snapshot, each extent Nlayer (ray: Nlayer-1 used), order of output()'s WRITEs */
typedef enum {
  SAMSIM_SNAPARR_T = 0, SAMSIM_SNAPARR_PSI_S, SAMSIM_SNAPARR_THICK, SAMSIM_SNAPARR_S_BU, SAMSIM_SNAPARR_RAY,
  SAMSIM_SNAPARR_PSI_L, SAMSIM_SNAPARR_PERM, SAMSIM_SNAPARR_FLUSH_V, SAMSIM_SNAPARR_FLUSH_H, SAMSIM_SNAPARR_PSI_G,
  /* rows of output_bgc (mo_output.f90:156-188): bulk and brine concentration per tracer; zero without tracers */
  SAMSIM_SNAPARR_BGC1_BU, SAMSIM_SNAPARR_BGC1_BR, SAMSIM_SNAPARR_BGC2_BU, SAMSIM_SNAPARR_BGC2_BR,
  SAMSIM_SNAPARR_COUNT
} samsim_snapshot_array_id;

/* ---- lifetime ---------------------------------------------------------------------------- */
/* Allocates device state for ncol columns on CUDA device `device`.  Arrays start zeroed like
 * sub_allocate (mo_init.f90:2082-2088).  Fails with SAMSIM_ERR_NO_DEVICE without a GPU. */
int samsim_b200_create(const samsim_config_t* cfg, int32_t ncol, int32_t device, samsim_handle_t* out);
void samsim_b200_destroy(samsim_handle_t h);
const char* samsim_b200_last_error(void);
const char* samsim_b200_version(void);

/* ---- state (mo_data) ---------------------------------------------------------------------- */
int32_t samsim_b200_array_extent(samsim_handle_t h, int32_t array_id);
int samsim_b200_set_array(samsim_handle_t h, int32_t array_id, const double* host, int32_t col0, int32_t n);
int samsim_b200_get_array(samsim_handle_t h, int32_t array_id, double* host, int32_t col0, int32_t n);
int samsim_b200_set_scalar(samsim_handle_t h, int32_t scalar_id, const double* host, int32_t col0, int32_t n);
int samsim_b200_get_scalar(samsim_handle_t h, int32_t scalar_id, double* host, int32_t col0, int32_t n);
int samsim_b200_set_int(samsim_handle_t h, int32_t int_id, const int32_t* host, int32_t col0, int32_t n);
int samsim_b200_get_int(samsim_handle_t h, int32_t int_id, int32_t* host, int32_t col0, int32_t n);
/* Replicate column `src` into columns [col0, col0+n): ensemble start from one initial state. */
int samsim_b200_broadcast_column(samsim_handle_t h, int32_t src, int32_t col0, int32_t n);

/* The clock is shared by the batch: time (mo_data.f90:59), loop index i of the LAST executed
 * step (0 before the first), n_time_out (:74), time_counter (:172, 1-based). */
int samsim_b200_set_clock(samsim_handle_t h, double time, int64_t i, int32_t n_time_out, int32_t time_counter);
int samsim_b200_get_clock(samsim_handle_t h, double* time, int64_t* i, int32_t* n_time_out, int32_t* time_counter);

/* ---- forcing ------------------------------------------------------------------------------ */
/* atmoflux_flag 2 (mo_functions.f90:304-327): nsite base sites, 4 series of nrec 3-hourly records
 * each, series[(site*4 + kind)*nrec + r]; time_input(k) = (k-1)*10800 s.  Column c reads site
 * site_of_col[c] through value*scale + offset with scale/offset[kind*ncol + c]; NULL = site 0 /
 * identity.  One multiply and one add in double, so the CPU oracle fed series*scale+offset
 * matches bit for bit.  Any nsite >= 1 is accepted, up to one site per column or more (a reanalysis grid cell per
 * column, or a series shifted in time per ensemble member for its own start date); only device memory limits the
 * table (nsite*4*nrec doubles).  Up to 16 sites are staged in shared memory per launch, larger tables are read in
 * place; both give the same results.  site_of_col is checked before anything is replaced (SAMSIM_ERR_ARG leaves the
 * previous forcing in place).  If a device allocation or copy fails (SAMSIM_ERR_CUDA), the handle holds no forcing
 * at all afterwards, as if set_forcing had never been called: steps with atmoflux_flag 2 return SAMSIM_ERR_STATE
 * until a set_forcing succeeds. */
int samsim_b200_set_forcing(samsim_handle_t h, int32_t nsite, int32_t nrec, const double* series,
                            const int32_t* site_of_col, const double* scale, const double* offset);
/* Refresh the base series of an existing forcing table in place (same nsite/nrec; per-column vectors are kept):
 * the streaming path when new reanalysis records arrive while the run is in progress.  Asynchronous on the handle's
 * stream when `series` is pinned host memory. */
int samsim_b200_update_forcing(samsim_handle_t h, const double* series);
/* Refresh records rec0 .. rec0+n-1 (1-based) of every site and kind of the table of the last set_forcing from
 * series[(site*4 + kind)*n + r], r = 0..n-1; all other records are kept.  The streaming path of large tables: a day
 * of new records for every site, without sending the whole table again.  One 2-D copy on the handle's stream,
 * ordered with launches like samsim_b200_update_forcing (asynchronous when `series` is pinned host memory).
 * SAMSIM_ERR_STATE before set_forcing; SAMSIM_ERR_ARG for a NULL pointer, n < 1 or records outside 1..nrec. */
int samsim_b200_update_forcing_records(samsim_handle_t h, int32_t rec0, int32_t n, const double* series);
/* Stochastic forcing perturbations: per-column AR(1) red noise on the records of the table, generated on the device
 * from a counter-based generator, so that a column's perturbation is a function of (seed, stream, kind, record) only
 * and does not depend on launch lengths, re-binning, shards or restarts.  Per kind k (samsim_forcing_kind order):
 * sigma[k] finite and >= 0 (0 leaves the kind untouched), phi[k] in [0, 1) (AR(1) coefficient per 3-hourly record),
 * mode[k] 0 additive, 1 multiplicative, 2 lognormal.  stream_of_col[c] in the caller's column order: columns with equal
 * ids get identical noise, -1 = unperturbed (control members); NULL = stream c.  All sigma 0 switches the feature off
 * (the default).  A bad argument (NaN, infinite or negative sigma, phi outside [0, 1), an unknown mode, a stream below
 * -1) is SAMSIM_ERR_ARG and keeps the previous setting; a config without atmoflux_flag 2 is SAMSIM_ERR_CONFIG; a failed
 * device allocation is SAMSIM_ERR_CUDA and leaves the feature off.  A run input like the table: not saved in
 * checkpoints.
 *
 * Bitwise contract.  For stream s >= 0, kind k and table record r >= 1:
 *   (x0,x1,x2,x3) = Philox4x32-10(counter = (r, k, s, 0), key = (seed & 0xffffffff, seed >> 32))   (Random123)
 *   u1 = ((double)(x0 >> 6) * 2^26 + (double)(x1 >> 6) + 0.5) * 2^-52,  u2 likewise from x2, x3
 *   z(r) = sqrt(-2.0 * det_log(u1)) * det_cos(6.283185307179586 * u2)
 *   e(1) = sigma * z(1);  e(r) = phi * e(r-1) + c * z(r),  c = sigma * sqrt(1.0 - phi * phi)
 * each operation rounded on its own; det_log / det_cos / det_exp are those of detmath.h.  The record value
 * v = base * scale + offset becomes v + e (additive), v * fmax(1.0 + e, 0.0) (multiplicative) or
 * v * det_exp(e - 0.5 * (sigma * sigma)) (lognormal, mean kept); stream -1 and sigma 0 read v unchanged.  Between
 * records the step interpolates the perturbed records linearly, as it does the plain ones.
 *
 * Device memory while on: SAMSIM_MAXWIN (24) * 4 * ncol_pad doubles for the perturbed records of a launch's window
 * (805 MB at 1,048,576 columns), 8 * ncol_pad doubles of recursion state and ncol int32 stream ids. */
int samsim_b200_set_stochastic_forcing(samsim_handle_t h, uint64_t seed, const double sigma[4], const double phi[4],
                                       const int32_t mode[4], const int32_t* stream_of_col);
/* The perturbation applied: out[c*nrec + r] = e(rec0 + r) of kind `kind` for the stream of caller column col0 + c
 * (records rec0 >= 1), 0 for stream -1, for sigma 0 and while the feature is off.  Computed on the device from the
 * definition, independent of the run. */
int samsim_b200_get_forcing_noise(samsim_handle_t h, int32_t kind, int32_t rec0, int32_t nrec, int32_t col0, int32_t n,
                                  double* out);
/* Correlated stochastic forcing: the four kinds drawn together and spatially coherent noise from shared basis streams.
 * A generalisation of samsim_b200_set_stochastic_forcing, which it replaces (and which replaces it): one setting, one
 * state.  sigma, phi, mode as there.  corr[16] (row-major, NULL = the identity) correlates the kinds' innovations: finite,
 * exactly symmetric, unit diagonal, positive definite.  Column c mixes nmix (1..8) basis streams:
 * basis_of_col[c*nmix + m] ids >= 0, distinct within the column, or -1 for an empty entry;
 * weight_of_col[c*nmix + m] finite weights (NULL = 1.0).  A column whose entries are all empty is unperturbed.
 *
 * Bitwise contract.  For basis stream b and record r, z_k(r; b) is z(r) of the single-stream contract with s = b, for
 * all four kinds.  w_k = z_k when corr is NULL or the identity, else w_k = ((L[k][0]*z_0 + L[k][1]*z_1) + ...) +
 * L[k][k]*z_k, L the Cholesky factor of corr by Cholesky-Banachiewicz in double (s = corr[i][j]; s = s - L[i][m]*L[j][m]
 * for m = 0..j-1; L[i][i] = sqrt(s), L[i][j] = s / L[j][j]).  E_k(1) = sigma_k * w_k(1), E_k(r) = phi_k * E_k(r-1) +
 * c_k * w_k(r).  Over a column's non-empty entries in m order, e = w * E(b) of the first, then e = e + w * E(b); the
 * modes read e, with h * q for the lognormal one, q = w*w of the first entry, then q = q + w*w.  So the lognormal mean is
 * kept, and nmix 1, weight 1.0 and the identity give the bits of samsim_b200_set_stochastic_forcing.  The lag-0
 * correlation of kinds i, j is corr[i][j] * sqrt((1-phi_i^2)(1-phi_j^2)) / (1 - phi_i*phi_j); two columns with unit-norm
 * weights correlate by the sum of w_a*w_b over their shared ids.  samsim_b200_get_forcing_noise returns the column's e.
 *
 * Errors as samsim_b200_set_stochastic_forcing; SAMSIM_ERR_ARG also for nmix outside 1..8, an id below -1, a repeated
 * id within a column, a non-finite weight, a bad corr or basis_of_col NULL.  Device memory while on: the window of
 * SAMSIM_MAXWIN * 4 * ncol_pad doubles, and, unless the setting is the single-stream case, SAMSIM_MAXWIN * 4 * nbasis +
 * 8 * nbasis doubles and 12 * nmix bytes per column (nbasis = the distinct ids) in place of the per-column state. */
int samsim_b200_set_stochastic_forcing_correlated(samsim_handle_t h, uint64_t seed, const double sigma[4],
                                                  const double phi[4], const int32_t mode[4], const double corr[16],
                                                  int32_t nmix, const int32_t* basis_of_col, const double* weight_of_col);
/* lab series (mo_grotz.f90:138-169): nset record sets of nrec per-dt values, kinds
 * 0 Tice->T2m, 1 snowfall->solid_precip, 2 heat->fl_q_bottom, 3 styropor; series[(set*4+kind)*nrec + r];
 * set_of_col NULL = set 0.  snow_precip_flag 0 zeroes the snowfall like the reference. */
int samsim_b200_set_lab_forcing(samsim_handle_t h, int32_t nset, int64_t nrec, const double* series,
                                const int32_t* set_of_col);
/* Real length of each lab set when the sets of one table differ in length (experiments of different durations):
 * the series stay padded to the nrec of samsim_b200_set_lab_forcing, and set s holds nrec_of_set[s] records
 * (1..nrec).  nset must be that of the last samsim_b200_set_lab_forcing, which resets every length to nrec.
 * samsim_b200_step checks each set whose columns have not all passed their end step against its own length. */
int samsim_b200_set_lab_lengths(samsim_handle_t h, int32_t nset, const int64_t* nrec_of_set);

/* ---- the hot path ------------------------------------------------------------------------- */
/* Advance every column nsteps iterations of mo_grotz.f90:182-835 (S0-S24 except the file I/O of
 * S6/S8; S8's accumulator averaging and reset are done on the device at the reference's cadence).
 * Columns whose status is non-zero are frozen, and so are columns past their end step.  With lab forcing, a
 * running column whose set would be read past its length makes the call return SAMSIM_ERR_STATE after the steps
 * that fit.  Asynchronous on the handle's stream. */
int samsim_b200_step(samsim_handle_t h, int64_t nsteps);
/* Per-column end step: column col0+q runs loop index i only while i <= end_i[q], so one batch can hold runs of
 * different lengths (time_total of each testcase, forcing records of each site).  A column past its end is frozen
 * like a failed one but keeps status 0; it writes no more S8 records, so its snapshot keeps the last record it wrote
 * (SAMSIM_SNAPSC_TIME says which).  Values must be >= 0 (else SAMSIM_ERR_ARG); INT64_MAX = no end, the default; an
 * end at or below the current i freezes the column from now on.  Caller's column numbering, like every setter. */
int samsim_b200_set_end_step(samsim_handle_t h, const int64_t* end_i, int32_t col0, int32_t n);
int samsim_b200_synchronize(samsim_handle_t h);
/* Steps from now until (and including) the next step that writes an output record. */
int64_t samsim_b200_steps_to_next_output(samsim_handle_t h);

/* ---- output at S8 ------------------------------------------------------------------------- */
int samsim_b200_set_snapshot_mode(samsim_handle_t h, int32_t mode);
/* values captured at the most recent output step; scalars[c*SAMSIM_SNAPSC_COUNT + id],
 * arrays[(c*SAMSIM_SNAPARR_COUNT + id)*Nlayer + (k-1)] (arrays may be NULL) */
int samsim_b200_get_snapshot(samsim_handle_t h, double* scalars, double* arrays, int32_t col0, int32_t n);

/* ---- ensemble statistics per column group at every S8 record ------------------------------------
 * Computed and kept on the device, so that one samsim_b200_step call may span any number of records.  ngroup = 0
 * switches them off (the default).  group_of_col[c] in [-1, ngroup) in the caller's column order, -1 = in no group,
 * NULL = every column in group 0.  depth[0..nz): metres below the ice surface (the top of layer 1), finite, > 0 and
 * strictly increasing; nz = 0 = scalars only.  profile_mask: bits of samsim_snapshot_array_id (not RAY; tracer rows only
 * with N_bgc tracers; non-zero needs nz > 0).  A bad argument is SAMSIM_ERR_ARG and keeps the previous setting; a
 * snapshot mode below SCALARS (FULL with profiles) is SAMSIM_ERR_STATE.  A new setting drops the held records.
 *
 * Quantities q: the SAMSIM_SNAPSC_COUNT scalars, then nz depths of each selected profile in samsim_snapshot_array_id
 * order.  stats[((r*ngroup + g)*Q + q)*5 + s], s = count, mean, variance, min, max; rec_time[r] = SAMSIM_SNAPSC_TIME
 * and rec_i[r] = loop index of record r; any output pointer may be NULL.
 *
 * Bitwise contract.  A member contributes to the record of step i when its status is 0 at the end of step i and its
 * end step is >= i.  Profile p at depth z: p(k) of the smallest k <= N_active with z <= D_k, D_k = (((thick(1) +
 * thick(2)) + ...) + thick(k)) over the snapshot; a member with z > D_{N_active} does not contribute there.  Sums are
 * the pairwise tree over ALL members of the group in ascending caller column order (non-contributing ones +0.0),
 * padded with +0.0 to a power of two, a = a[0::2] + a[1::2] repeated; mean = S / count; M2 = the same tree over
 * (x - mean)^2 (+0.0 for the others); variance = M2 / (count - 1), 0 for count 1; min / max = fmin / fmax over the
 * contributors; count 0 gives NaN for mean, variance, min and max.  Results do not depend on re-binning or launch
 * lengths.
 *
 * samsim_b200_step with statistics on: no launch runs past an output step, and after each launch that ends on one the
 * statistics kernels are queued on the handle's stream (no host synchronisation).  A call that would write more
 * records than max_records - held returns SAMSIM_ERR_STATE before anything runs.  Not saved in checkpoints. */
int samsim_b200_set_group_stats(samsim_handle_t h, int32_t ngroup, const int32_t* group_of_col, int32_t nz,
                                const double* depth, uint32_t profile_mask, int32_t max_records);
int32_t samsim_b200_group_stats_held(samsim_handle_t h); /* records held, -1 for a null handle */
int samsim_b200_get_group_stats(samsim_handle_t h, double* stats, double* rec_time, int64_t* rec_i, int32_t rec0,
                                int32_t nrec);
int samsim_b200_clear_group_stats(samsim_handle_t h); /* drop the held records */

/* ---- per-column time statistics over windows of S8 records ----------------------------------------
 * Accumulated and kept on the device, so that one samsim_b200_step call may span any number of records and windows.
 * Quantities q: the SAMSIM_SNAPSC_* scalars whose bits are set in scalar_mask (bits 0..19), in id order, then nz
 * depths of each profile selected by profile_mask in samsim_snapshot_array_id order; Q = their number.  depth and
 * profile_mask follow the rules of samsim_b200_set_group_stats (finite, > 0, strictly increasing; not RAY; tracer
 * rows only with N_bgc tracers; non-zero needs nz > 0).  Q = 0 (both masks 0) switches them off (the default).  A bad
 * argument is SAMSIM_ERR_ARG and keeps the previous setting; a snapshot mode below SCALARS (FULL with profiles) is
 * SAMSIM_ERR_STATE.  A new setting drops the held windows and the window in progress.  Device memory:
 * (1 + max_windows) * 5 * Q * ncol_pad doubles; a failed allocation is SAMSIM_ERR_CUDA and leaves them off.
 *
 * Windows: a window collects records_per_window (>= 0) consecutive records, counted from the set call or the last
 * close; its last record finalises it into history slot `held` and a new window starts.  records_per_window = 0: a
 * window closes only through samsim_b200_close_time_window (calendar windows such as months).  Closing an empty
 * window, or closing with a full history, is SAMSIM_ERR_STATE.
 *
 * Output for windows win0..win0+nwin-1 and caller columns col0..col0+n-1: stats[((w*n + c)*Q + q)*5 + s], s = count,
 * mean, variance, min, max; win_nrec[w] = records in window w; win_time[2w], [2w+1] = SAMSIM_SNAPSC_TIME and win_i[2w],
 * [2w+1] = loop index of its first and last record; any output pointer may be NULL.
 *
 * Bitwise contract.  A column contributes the record of step i when its status is 0 at the end of step i and its end
 * step is >= i.  Profile p at depth z takes the layer of samsim_b200_set_group_stats' regrid; depths below D_{N_active}
 * do not contribute, so every quantity has its own count.  Records are accumulated in record order, starting from
 * n = 0, mean = 0, M2 = 0, min = max = NaN, with exactly
 *     n = n + 1;  d = x - mean;  mean = mean + d / n;  M2 = M2 + d * (x - mean);  min = fmin(min, x);  max = fmax(max, x)
 * (no contraction; of two equal values, +0.0 and -0.0, fmin / fmax keep min / max).  Finalising: mean NaN for count 0;
 * variance = M2 / (n - 1), 0 for n = 1, NaN for n = 0; min and max NaN for count 0.  Results do not depend on
 * re-binning, launch lengths, block size, the two-pass step or whether group statistics are on.
 *
 * samsim_b200_step with time statistics on: no launch runs past an output step, and after each launch that ends on one
 * the time-statistics kernel is queued on the handle's stream (no host synchronisation).  A call that would complete
 * more windows than max_windows - held returns SAMSIM_ERR_STATE before anything runs.  Time statistics are run outputs:
 * not saved in checkpoints; samsim_b200_load_checkpoint and samsim_b200_set_clock leave the accumulators alone. */
int samsim_b200_set_time_stats(samsim_handle_t h, int32_t records_per_window, uint32_t scalar_mask, int32_t nz,
                               const double* depth, uint32_t profile_mask, int32_t max_windows);
int32_t samsim_b200_time_stats_held(samsim_handle_t h); /* completed windows held, -1 for a null handle */
int samsim_b200_get_time_stats(samsim_handle_t h, double* stats, int32_t* win_nrec, double* win_time, int64_t* win_i,
                               int32_t win0, int32_t nwin, int32_t col0, int32_t n);
int samsim_b200_close_time_window(samsim_handle_t h); /* close the window in progress now */
int samsim_b200_clear_time_stats(samsim_handle_t h);  /* drop the held windows */

/* ---- diagnostics -------------------------------------------------------------------------- */
int samsim_b200_get_status(samsim_handle_t h, int32_t* status, int32_t col0, int32_t n);
/* number of columns with non-zero status */
int samsim_b200_count_failed(samsim_handle_t h, int32_t* nfailed);
/* sum/min/max over this device's columns of SAMSIM_SNAPSC_* style diagnostics computed from the
 * current state: out[3*j + {0,1,2}] for j in {thickness, bulk_salin, freeboard, thick_snow, T_top, N_active}.
 * The multi-GPU reduction of these 18 numbers is one NCCL all-reduce in the host layer. */
int samsim_b200_reduce_diag(samsim_handle_t h, double* out18);
/* kernel launches issued by this handle so far (bench.py's gpu_launches) */
int64_t samsim_b200_launch_count(samsim_handle_t h);
/* time (ms) of the last samsim_b200_step measured with CUDA events on the handle's stream */
int samsim_b200_last_step_ms(samsim_handle_t h, float* ms);
/* ---- re-binning (SURVEY 8e: "within a GPU, columns are periodically re-binned by N_active / snow regime for
 * warp coherence; local permutation only, an index array maps back") ---------------------------
 * The reference has one column per process, so there is nothing to replace: this is what a batch needs so that
 * columns whose N_active (loop trip counts, mo_grotz.f90:298-307,592-598) and snow branches (mo_grotz.f90:273-292)
 * differ do not share a warp.  Results do not depend on it (columns are independent); every entry point keeps
 * taking the caller's column numbers.  *changed = 1 if the device order changed. */
int samsim_b200_rebin(samsim_handle_t h, int32_t* changed);
/* Kernel tuning; results do not depend on it (bitwise, tests/test_parity_gpu.py runs both settings).
 * two_pass = 1: columns in a steady regime (no flooding, flushing or layer event, a snow layer of its own or no snow)
 * advance a step in two sweeps over their layers -- S4..S17 merged into one forward pass, S18 plus the next step's
 * Rayleigh-number estimates in one backward pass (DESIGN.md section 5) -- 21 array passes per step instead of 34 and
 * 30 % less DRAM traffic; the general sub-step-by-sub-step path (two_pass = 0, the default) is currently the faster
 * one on B200 because the merged pass is register-starved at 64 registers per thread. */
/* prefetch_layers: L1 prefetch distance of the layer sweeps (0 = keep the default of 2). */
int samsim_b200_set_tuning(samsim_handle_t h, int32_t two_pass, int32_t prefetch_layers);
/* re-bin automatically every nsteps steps inside samsim_b200_step (0 = never, the default) */
int samsim_b200_set_rebin_interval(samsim_handle_t h, int64_t nsteps);
/* Divergence-driven re-binning.  At the end of every launch each warp of the step kernel measures its own divergence
 * with warp reductions and ballots: idle lane-layers = SUM over lanes of (deepest N_active in the warp - the lane's
 * N_active) against all lane-layers, and whether its lanes disagree on the regime class: the snow class (no snow /
 * traces / thin, coupled to layer 1 / a layer of its own) and whether the surface melted in the last step (such a
 * column flushes and re-solves every layer in the next step; one such lane makes its warp pay for both).  With a
 * threshold > 0 the next samsim_b200_step re-bins the columns first when the idle share of the previous launch
 * exceeded it (or more than four times that share of warps were split by class); 0 switches the automatic mode off
 * (the default).  Re-binning sorts by (failed, N_active descending, class, forcing site, surface temperature in 0.1 K buckets). */
int samsim_b200_set_rebin_auto(samsim_handle_t h, double idle_share_threshold);
/* the last launch's measurement (waits for it), and the number of re-binnings so far; any pointer may be NULL */
int samsim_b200_get_divergence(samsim_handle_t h, double* idle_lane_layer_share, double* snow_class_split_warp_share,
                               int64_t* rebins);
/* slot_of_col[c] = position of column c in the device arrays (identity until the first re-binning) */
int samsim_b200_get_slot_map(samsim_handle_t h, int32_t* slot_of_col);

/* ---- checkpoint / restart (SURVEY 8f-4) ------------------------------------------------------
 * The reference can only start from init(testcase) (mo_init.f90:62); a year of 1 M columns wants restarts.
 * save: every state array, scalar and int of every column plus the clock, in the caller's column order.
 * load: into a handle created with the same config and column count (else SAMSIM_ERR_CONFIG); forcing tables, end
 * steps and lab lengths are run inputs and must be set again.  A restarted run continues bit-identically. */
int samsim_b200_save_checkpoint(samsim_handle_t h, const char* path);
int samsim_b200_load_checkpoint(samsim_handle_t h, const char* path);

/* raw device pointers for zero-copy interop (torch).  arrays is the warp-tiled state buffer
 * arrays[ncol_pad/32][lstride][narrays][32]: element (array a, layer k = 0..Nlayer+1) of the column in device slot s is
 * arrays[(((s/32)*lstride + k)*narrays + a)*32 + s%32]; a = samsim_array_id for the first 15 arrays, the tracer arrays
 * sit at a = 22, 23 (behind the scratch arrays).  scalars[scalar_id][ncol_pad], ints[int_id][ncol_pad].  The column
 * index is the SLOT (samsim_b200_get_slot_map) once the handle has been re-binned. */
int samsim_b200_device_layout(samsim_handle_t h, void** arrays, void** scalars, void** ints, int64_t* ncol_pad,
                              int64_t* lstride, int64_t* narrays);

/* ---- unit known-answer entry points (device functions evaluated elementwise on the GPU) ---- */
/* status_out[q]: STOP code (0 or 99) in the low 16 bits, the SAMSIM_EV_GETT_* bits of event word 1 shifted left by 16 */
int samsim_b200_kat_getT(int32_t salt_flag, int32_t n, const double* H, const double* S_bu, const double* T_in,
                         double* T_out, double* phi_out, int32_t* status_out, int32_t device);
/* fn: 0 S_br(a) 1 S_br(a,b) 2 ddT_S_br(a) 3 density(a,b) 4 T_freeze(a) 5 k_snow(a,b) 6 albedo(a,b)
 *     7 det_pow(a,b) 8 det_exp(a) 9 det_sin(a) */
int samsim_b200_kat_scalar(int32_t fn, int32_t salt_flag, int32_t n, const double* a, const double* b, double* out,
                           int32_t device);
/* FP64 peak microbenchmark: dependent-free DFMA chains on all SMs; returns achieved TFLOP/s */
int samsim_b200_fp64_peak(int32_t device, double seconds, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* SAMSIM_B200_H */
