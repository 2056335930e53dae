!>
!! ISO_C_BINDING interface to the B200 column-timestep library (include/samsim_b200.h).
!!
!! This module is the reference-side binding a SAMSIM maintainer adds next to mo_grotz.f90.  It declares the C
!! entry points, mirrors samsim_config_t as a BIND(C) type, and provides pack/unpack helpers between the
!! module-global state of mo_data (mo_data.f90:34-203) and the device.  mo_grotz_b200.f90 uses it to replace the
!! body of `DO i = 1,i_time` (mo_grotz.f90:182-835).
!!
!! NOTE: this image has no Fortran compiler (gfortran/f951, flang, nvfortran are absent), so this file is shipped
!! uncompiled; the same ABI is exercised by samsim_b200/api.py (ctypes) in the test-suite.
!!
MODULE mo_samsim_b200

  USE, INTRINSIC :: ISO_C_BINDING
  IMPLICIT NONE
  PUBLIC

  !> samsim_config_t: 26 x int32 then 10 x double (tests/test_cabi_cpu.py::test_config_struct_layout)
  TYPE, BIND(C) :: samsim_config_t
     INTEGER(C_INT32_T) :: testcase
     INTEGER(C_INT32_T) :: Nlayer, N_top, N_middle, N_bottom
     INTEGER(C_INT32_T) :: atmoflux_flag, grav_flag, prescribe_flag, grav_heat_flag, flush_heat_flag, turb_flag, &
          &                salt_flag, boundflux_flag, flush_flag, flood_flag, bottom_flag, precip_flag, harmonic_flag, &
          &                tank_flag, albedo_flag, lab_snow_flag, freeboard_snow_flag, snow_flush_flag, snow_precip_flag
     INTEGER(C_INT32_T) :: i_time_out
     INTEGER(C_INT32_T) :: N_bgc
     REAL(C_DOUBLE)     :: dt, thick_0, thick_min, time_out
     REAL(C_DOUBLE)     :: alpha_flux_instable, alpha_flux_stable
     REAL(C_DOUBLE)     :: m_total
     REAL(C_DOUBLE)     :: max_flux_plate, k_snow_flush, k_styropor
  END TYPE samsim_config_t

  ! samsim_array_id
  INTEGER(C_INT32_T), PARAMETER :: SAMSIM_ARR_M = 0, SAMSIM_ARR_S_ABS = 1, SAMSIM_ARR_H_ABS = 2, SAMSIM_ARR_THICK = 3, &
       & SAMSIM_ARR_T = 4, SAMSIM_ARR_PHI = 5, SAMSIM_ARR_S_BU = 6, SAMSIM_ARR_PSI_S = 7, SAMSIM_ARR_PSI_L = 8, &
       & SAMSIM_ARR_PSI_G = 9, SAMSIM_ARR_RAY = 10, SAMSIM_ARR_PERM = 11, SAMSIM_ARR_FLUSH_V = 12, &
       & SAMSIM_ARR_FLUSH_H = 13, SAMSIM_ARR_FL_Q = 14, SAMSIM_ARR_BGC_ABS1 = 15, SAMSIM_ARR_BGC_ABS2 = 16
  ! samsim_scalar_id (order of include/samsim_b200.h)
  INTEGER(C_INT32_T), PARAMETER :: SC_T_BOTTOM = 0, SC_T_TOP = 1, SC_S_BU_BOTTOM = 2, SC_T2M = 3, SC_FL_Q_BOTTOM = 4, &
       & SC_PSI_S_SNOW = 5, SC_PSI_L_SNOW = 6, SC_PSI_G_SNOW = 7, SC_PHI_S = 8, SC_S_ABS_SNOW = 9, SC_H_ABS_SNOW = 10, &
       & SC_M_SNOW = 11, SC_T_SNOW = 12, SC_THICK_SNOW = 13, SC_LIQUID_PRECIP = 14, SC_SOLID_PRECIP = 15, &
       & SC_FL_Q_SNOW = 16, SC_ENERGY_STORED = 17, SC_TOTAL_RESIST = 18, SC_FRESHWATER = 19, SC_THICKNESS = 20, &
       & SC_BULK_SALIN = 21, SC_ALBEDO = 22, SC_FL_SW = 23, SC_FL_LW = 24, SC_FL_REST = 25, SC_GRAV_DRAIN = 26, &
       & SC_GRAV_SALT = 27, SC_GRAV_TEMP = 28, SC_MELT_THICK = 29, SC_MELT_THICK_SNOW = 30, &
       & SC_MELT_THICK_SNOW_OLD = 31, SC_MTO1 = 32, SC_MTO2 = 33, SC_MTO3 = 34, SC_FREEBOARD = 35, SC_T_FREEZE = 36, &
       & SC_MELT_ERR = 37, SC_S_TOTAL = 38, SC_TTOP_WARM = 39, SC_TTOP_COLD = 40, SC_OFLUX_AMP = 41, &
       & SC_BGC_BOTTOM1 = 42, SC_BGC_BOTTOM2 = 43, SC_BGC_TOTAL1 = 44, SC_BGC_TOTAL2 = 45
  INTEGER(C_INT32_T), PARAMETER :: SAMSIM_INT_N_ACTIVE = 0, SAMSIM_INT_STATUS = 1, SAMSIM_INT_STYROPOR_FLAG = 2
  INTEGER(C_INT32_T), PARAMETER :: SAMSIM_SNAP_NONE = 0, SAMSIM_SNAP_SCALARS = 1, SAMSIM_SNAP_FULL = 2

  INTERFACE
     INTEGER(C_INT) FUNCTION samsim_b200_create(cfg, ncol, device, handle) BIND(C, NAME='samsim_b200_create')
       IMPORT :: C_INT, C_INT32_T, C_PTR, samsim_config_t
       TYPE(samsim_config_t), INTENT(in) :: cfg
       INTEGER(C_INT32_T), VALUE :: ncol, device
       TYPE(C_PTR), INTENT(out) :: handle
     END FUNCTION samsim_b200_create

     SUBROUTINE samsim_b200_destroy(handle) BIND(C, NAME='samsim_b200_destroy')
       IMPORT :: C_PTR
       TYPE(C_PTR), VALUE :: handle
     END SUBROUTINE samsim_b200_destroy

     INTEGER(C_INT) FUNCTION samsim_b200_set_array(handle, id, host, col0, n) BIND(C, NAME='samsim_b200_set_array')
       IMPORT :: C_INT, C_INT32_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: id, col0, n
       REAL(C_DOUBLE), INTENT(in) :: host(*)
     END FUNCTION samsim_b200_set_array

     INTEGER(C_INT) FUNCTION samsim_b200_get_array(handle, id, host, col0, n) BIND(C, NAME='samsim_b200_get_array')
       IMPORT :: C_INT, C_INT32_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: id, col0, n
       REAL(C_DOUBLE), INTENT(out) :: host(*)
     END FUNCTION samsim_b200_get_array

     INTEGER(C_INT) FUNCTION samsim_b200_set_scalar(handle, id, host, col0, n) BIND(C, NAME='samsim_b200_set_scalar')
       IMPORT :: C_INT, C_INT32_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: id, col0, n
       REAL(C_DOUBLE), INTENT(in) :: host(*)
     END FUNCTION samsim_b200_set_scalar

     INTEGER(C_INT) FUNCTION samsim_b200_get_scalar(handle, id, host, col0, n) BIND(C, NAME='samsim_b200_get_scalar')
       IMPORT :: C_INT, C_INT32_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: id, col0, n
       REAL(C_DOUBLE), INTENT(out) :: host(*)
     END FUNCTION samsim_b200_get_scalar

     INTEGER(C_INT) FUNCTION samsim_b200_set_int(handle, id, host, col0, n) BIND(C, NAME='samsim_b200_set_int')
       IMPORT :: C_INT, C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: id, col0, n
       INTEGER(C_INT32_T), INTENT(in) :: host(*)
     END FUNCTION samsim_b200_set_int

     INTEGER(C_INT) FUNCTION samsim_b200_get_int(handle, id, host, col0, n) BIND(C, NAME='samsim_b200_get_int')
       IMPORT :: C_INT, C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: id, col0, n
       INTEGER(C_INT32_T), INTENT(out) :: host(*)
     END FUNCTION samsim_b200_get_int

     INTEGER(C_INT) FUNCTION samsim_b200_broadcast_column(handle, src, col0, n) BIND(C, NAME='samsim_b200_broadcast_column')
       IMPORT :: C_INT, C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: src, col0, n
     END FUNCTION samsim_b200_broadcast_column

     INTEGER(C_INT) FUNCTION samsim_b200_set_clock(handle, time, i, n_time_out, time_counter) BIND(C, NAME='samsim_b200_set_clock')
       IMPORT :: C_INT, C_INT32_T, C_INT64_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       REAL(C_DOUBLE), VALUE :: time
       INTEGER(C_INT64_T), VALUE :: i
       INTEGER(C_INT32_T), VALUE :: n_time_out, time_counter
     END FUNCTION samsim_b200_set_clock

     INTEGER(C_INT) FUNCTION samsim_b200_get_clock(handle, time, i, n_time_out, time_counter) BIND(C, NAME='samsim_b200_get_clock')
       IMPORT :: C_INT, C_INT32_T, C_INT64_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       REAL(C_DOUBLE), INTENT(out) :: time
       INTEGER(C_INT64_T), INTENT(out) :: i
       INTEGER(C_INT32_T), INTENT(out) :: n_time_out, time_counter
     END FUNCTION samsim_b200_get_clock

     INTEGER(C_INT) FUNCTION samsim_b200_set_forcing(handle, nsite, nrec, series, site_of_col, scale, offset) &
          & BIND(C, NAME='samsim_b200_set_forcing')
       IMPORT :: C_INT, C_INT32_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: nsite, nrec
       REAL(C_DOUBLE), INTENT(in) :: series(*)
       TYPE(C_PTR), VALUE :: site_of_col, scale, offset   !< C_NULL_PTR = site 0 / identity
     END FUNCTION samsim_b200_set_forcing

     !> refresh records rec0 .. rec0+n-1 (1-based) of every site and kind from series((site*4 + kind)*n + r)
     INTEGER(C_INT) FUNCTION samsim_b200_update_forcing_records(handle, rec0, n, series) &
          & BIND(C, NAME='samsim_b200_update_forcing_records')
       IMPORT :: C_INT, C_INT32_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: rec0, n
       REAL(C_DOUBLE), INTENT(in) :: series(*)
     END FUNCTION samsim_b200_update_forcing_records

     INTEGER(C_INT) FUNCTION samsim_b200_set_lab_forcing(handle, nset, nrec, series, set_of_col) &
          & BIND(C, NAME='samsim_b200_set_lab_forcing')
       IMPORT :: C_INT, C_INT32_T, C_INT64_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: nset
       INTEGER(C_INT64_T), VALUE :: nrec
       REAL(C_DOUBLE), INTENT(in) :: series(*)
       TYPE(C_PTR), VALUE :: set_of_col
     END FUNCTION samsim_b200_set_lab_forcing

     !> real length of each lab set when the sets are padded to one nrec (experiments of different durations)
     INTEGER(C_INT) FUNCTION samsim_b200_set_lab_lengths(handle, nset, nrec_of_set) &
          & BIND(C, NAME='samsim_b200_set_lab_lengths')
       IMPORT :: C_INT, C_INT32_T, C_INT64_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: nset
       INTEGER(C_INT64_T), INTENT(in) :: nrec_of_set(*)
     END FUNCTION samsim_b200_set_lab_lengths

     INTEGER(C_INT) FUNCTION samsim_b200_step(handle, nsteps) BIND(C, NAME='samsim_b200_step')
       IMPORT :: C_INT, C_INT64_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT64_T), VALUE :: nsteps
     END FUNCTION samsim_b200_step

     !> last loop index i of columns col0 .. col0+n-1 (0-based); HUGE(0_C_INT64_T) = no end
     INTEGER(C_INT) FUNCTION samsim_b200_set_end_step(handle, end_i, col0, n) BIND(C, NAME='samsim_b200_set_end_step')
       IMPORT :: C_INT, C_INT32_T, C_INT64_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT64_T), INTENT(in) :: end_i(*)
       INTEGER(C_INT32_T), VALUE :: col0, n
     END FUNCTION samsim_b200_set_end_step

     INTEGER(C_INT) FUNCTION samsim_b200_synchronize(handle) BIND(C, NAME='samsim_b200_synchronize')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: handle
     END FUNCTION samsim_b200_synchronize

     INTEGER(C_INT64_T) FUNCTION samsim_b200_steps_to_next_output(handle) BIND(C, NAME='samsim_b200_steps_to_next_output')
       IMPORT :: C_INT64_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
     END FUNCTION samsim_b200_steps_to_next_output

     INTEGER(C_INT) FUNCTION samsim_b200_set_snapshot_mode(handle, mode) BIND(C, NAME='samsim_b200_set_snapshot_mode')
       IMPORT :: C_INT, C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), VALUE :: mode
     END FUNCTION samsim_b200_set_snapshot_mode

     INTEGER(C_INT) FUNCTION samsim_b200_get_snapshot(handle, scalars, arrays, col0, n) BIND(C, NAME='samsim_b200_get_snapshot')
       IMPORT :: C_INT, C_INT32_T, C_PTR, C_DOUBLE
       TYPE(C_PTR), VALUE :: handle
       REAL(C_DOUBLE), INTENT(out) :: scalars(*), arrays(*)
       INTEGER(C_INT32_T), VALUE :: col0, n
     END FUNCTION samsim_b200_get_snapshot

     !> ensemble statistics per column group at every output record (ngroup = 0: off); group_of_col, depth: C_LOC of
     !> the arrays or C_NULL_PTR; profile_mask: bits of samsim_snapshot_array_id (uint32_t in C, masks < 2**14)
     INTEGER(C_INT) FUNCTION samsim_b200_set_group_stats(handle, ngroup, group_of_col, nz, depth, profile_mask, &
          & max_records) BIND(C, NAME='samsim_b200_set_group_stats')
       IMPORT :: C_INT, C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle, group_of_col, depth
       INTEGER(C_INT32_T), VALUE :: ngroup, nz, profile_mask, max_records
     END FUNCTION samsim_b200_set_group_stats

     INTEGER(C_INT32_T) FUNCTION samsim_b200_group_stats_held(handle) BIND(C, NAME='samsim_b200_group_stats_held')
       IMPORT :: C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
     END FUNCTION samsim_b200_group_stats_held

     !> records rec0 .. rec0+nrec-1 (0-based): stats(5, Q, ngroup, nrec), rec_time(nrec), rec_i(nrec); C_NULL_PTR skips one
     INTEGER(C_INT) FUNCTION samsim_b200_get_group_stats(handle, stats, rec_time, rec_i, rec0, nrec) &
          & BIND(C, NAME='samsim_b200_get_group_stats')
       IMPORT :: C_INT, C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle, stats, rec_time, rec_i
       INTEGER(C_INT32_T), VALUE :: rec0, nrec
     END FUNCTION samsim_b200_get_group_stats

     INTEGER(C_INT) FUNCTION samsim_b200_clear_group_stats(handle) BIND(C, NAME='samsim_b200_clear_group_stats')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: handle
     END FUNCTION samsim_b200_clear_group_stats

     !> per-column time statistics over windows of output records (both masks 0: off); depth: C_LOC of the array or
     !> C_NULL_PTR; scalar_mask: bits of samsim_snapshot_scalar_id, profile_mask: bits of samsim_snapshot_array_id
     !> (uint32_t in C, masks < 2**20)
     INTEGER(C_INT) FUNCTION samsim_b200_set_time_stats(handle, records_per_window, scalar_mask, nz, depth, &
          & profile_mask, max_windows) BIND(C, NAME='samsim_b200_set_time_stats')
       IMPORT :: C_INT, C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle, depth
       INTEGER(C_INT32_T), VALUE :: records_per_window, scalar_mask, nz, profile_mask, max_windows
     END FUNCTION samsim_b200_set_time_stats

     INTEGER(C_INT32_T) FUNCTION samsim_b200_time_stats_held(handle) BIND(C, NAME='samsim_b200_time_stats_held')
       IMPORT :: C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
     END FUNCTION samsim_b200_time_stats_held

     !> windows win0 .. win0+nwin-1 and columns col0 .. col0+n-1 (0-based): stats(5, Q, n, nwin), win_nrec(nwin),
     !> win_time(2, nwin), win_i(2, nwin); C_NULL_PTR skips one
     INTEGER(C_INT) FUNCTION samsim_b200_get_time_stats(handle, stats, win_nrec, win_time, win_i, win0, nwin, col0, n) &
          & BIND(C, NAME='samsim_b200_get_time_stats')
       IMPORT :: C_INT, C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle, stats, win_nrec, win_time, win_i
       INTEGER(C_INT32_T), VALUE :: win0, nwin, col0, n
     END FUNCTION samsim_b200_get_time_stats

     INTEGER(C_INT) FUNCTION samsim_b200_close_time_window(handle) BIND(C, NAME='samsim_b200_close_time_window')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: handle
     END FUNCTION samsim_b200_close_time_window

     INTEGER(C_INT) FUNCTION samsim_b200_clear_time_stats(handle) BIND(C, NAME='samsim_b200_clear_time_stats')
       IMPORT :: C_INT, C_PTR
       TYPE(C_PTR), VALUE :: handle
     END FUNCTION samsim_b200_clear_time_stats

     INTEGER(C_INT) FUNCTION samsim_b200_get_status(handle, status, col0, n) BIND(C, NAME='samsim_b200_get_status')
       IMPORT :: C_INT, C_INT32_T, C_PTR
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), INTENT(out) :: status(*)
       INTEGER(C_INT32_T), VALUE :: col0, n
     END FUNCTION samsim_b200_get_status

     ! batch-only helpers (nothing in the reference to replace): re-binning of drifted ensembles, restart files
     INTEGER(C_INT) FUNCTION samsim_b200_rebin(handle, changed) BIND(C, NAME='samsim_b200_rebin')
       IMPORT :: C_PTR, C_INT, C_INT32_T
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT32_T), INTENT(out) :: changed
     END FUNCTION samsim_b200_rebin

     INTEGER(C_INT) FUNCTION samsim_b200_set_rebin_interval(handle, nsteps) BIND(C, NAME='samsim_b200_set_rebin_interval')
       IMPORT :: C_PTR, C_INT, C_INT64_T
       TYPE(C_PTR), VALUE :: handle
       INTEGER(C_INT64_T), VALUE :: nsteps
     END FUNCTION samsim_b200_set_rebin_interval

     INTEGER(C_INT) FUNCTION samsim_b200_save_checkpoint(handle, path) BIND(C, NAME='samsim_b200_save_checkpoint')
       IMPORT :: C_PTR, C_INT, C_CHAR
       TYPE(C_PTR), VALUE :: handle
       CHARACTER(KIND=C_CHAR), DIMENSION(*), INTENT(in) :: path      ! NUL-terminated
     END FUNCTION samsim_b200_save_checkpoint

     INTEGER(C_INT) FUNCTION samsim_b200_load_checkpoint(handle, path) BIND(C, NAME='samsim_b200_load_checkpoint')
       IMPORT :: C_PTR, C_INT, C_CHAR
       TYPE(C_PTR), VALUE :: handle
       CHARACTER(KIND=C_CHAR), DIMENSION(*), INTENT(in) :: path
     END FUNCTION samsim_b200_load_checkpoint

     FUNCTION samsim_b200_last_error() BIND(C, NAME='samsim_b200_last_error') RESULT(msg)
       IMPORT :: C_PTR
       TYPE(C_PTR) :: msg
     END FUNCTION samsim_b200_last_error
  END INTERFACE

CONTAINS

  !> Abort like the reference does (`STOP <code>`) when a library call fails.
  SUBROUTINE b200_check(rc, what)
    INTEGER(C_INT), INTENT(in) :: rc
    CHARACTER(*),   INTENT(in) :: what
    IF (rc /= 0) THEN
       PRINT*, 'samsim_b200 call failed: ', what, rc
       STOP 4242
    END IF
  END SUBROUTINE b200_check

  !> Re-raises a reference STOP code reported by the device for the drop-in column (STOP needs a constant in
  !> Fortran 2003, hence the SELECT over the codes the path can raise; SURVEY section 4).
  SUBROUTINE b200_stop_with(code)
    INTEGER, INTENT(in) :: code
    SELECT CASE (code)
    CASE (99);    STOP 99
    CASE (98);    STOP 98
    CASE (16);    STOP 16
    CASE (345);   STOP 345
    CASE (9876);  STOP 9876
    CASE (21234); STOP 21234
    CASE (1337);  STOP 1337
    CASE (431);   STOP 431
    CASE (7889);  STOP 7889
    CASE DEFAULT; STOP 1
    END SELECT
  END SUBROUTINE b200_stop_with

  !> Builds samsim_config_t from the flags and scalars init() left in mo_data (mo_init.f90:83-132, :1982-2009).
  FUNCTION b200_config_from_mo_data(testcase) RESULT(cfg)
    USE mo_data
    USE mo_parameters, ONLY: max_flux_plate, k_snow_flush, k_styropor
    INTEGER, INTENT(in)   :: testcase
    TYPE(samsim_config_t) :: cfg
    cfg%testcase = testcase
    cfg%Nlayer = Nlayer;  cfg%N_top = N_top;  cfg%N_middle = N_middle;  cfg%N_bottom = N_bottom
    cfg%atmoflux_flag = atmoflux_flag;  cfg%grav_flag = grav_flag;  cfg%prescribe_flag = prescribe_flag
    cfg%grav_heat_flag = grav_heat_flag;  cfg%flush_heat_flag = flush_heat_flag;  cfg%turb_flag = turb_flag
    cfg%salt_flag = salt_flag;  cfg%boundflux_flag = boundflux_flag;  cfg%flush_flag = flush_flag
    cfg%flood_flag = flood_flag;  cfg%bottom_flag = bottom_flag;  cfg%precip_flag = precip_flag
    cfg%harmonic_flag = harmonic_flag;  cfg%tank_flag = tank_flag;  cfg%albedo_flag = albedo_flag
    cfg%lab_snow_flag = lab_snow_flag;  cfg%freeboard_snow_flag = freeboard_snow_flag
    cfg%snow_flush_flag = snow_flush_flag;  cfg%snow_precip_flag = snow_precip_flag
    cfg%i_time_out = i_time_out;  cfg%N_bgc = MERGE(N_bgc, 0, bgc_flag == 2)
    cfg%dt = dt;  cfg%thick_0 = thick_0;  cfg%thick_min = thick_min;  cfg%time_out = time_out
    cfg%alpha_flux_instable = alpha_flux_instable;  cfg%alpha_flux_stable = alpha_flux_stable
    cfg%m_total = m_total
    cfg%max_flux_plate = max_flux_plate;  cfg%k_snow_flush = k_snow_flush;  cfg%k_styropor = k_styropor
  END FUNCTION b200_config_from_mo_data

  SUBROUTINE put_sc(h, id, v)
    TYPE(C_PTR), INTENT(in) :: h
    INTEGER(C_INT32_T), INTENT(in) :: id
    REAL(C_DOUBLE), INTENT(in) :: v
    REAL(C_DOUBLE) :: buf(1)
    buf(1) = v
    CALL b200_check(samsim_b200_set_scalar(h, id, buf, 0_C_INT32_T, 1_C_INT32_T), 'set_scalar')
  END SUBROUTINE put_sc

  SUBROUTINE get_sc(h, id, v)
    TYPE(C_PTR), INTENT(in) :: h
    INTEGER(C_INT32_T), INTENT(in) :: id
    REAL(C_DOUBLE), INTENT(out) :: v
    REAL(C_DOUBLE) :: buf(1)
    CALL b200_check(samsim_b200_get_scalar(h, id, buf, 0_C_INT32_T, 1_C_INT32_T), 'get_scalar')
    v = buf(1)
  END SUBROUTINE get_sc

  !> mo_data -> device column 0 (then samsim_b200_broadcast_column replicates it for an ensemble).
  SUBROUTINE b200_push_mo_data(h)
    USE mo_data
    TYPE(C_PTR), INTENT(in) :: h
    INTEGER(C_INT32_T) :: ibuf(1)
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_M,       m,       0_C_INT32_T, 1_C_INT32_T), 'm')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_S_ABS,   S_abs,   0_C_INT32_T, 1_C_INT32_T), 'S_abs')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_H_ABS,   H_abs,   0_C_INT32_T, 1_C_INT32_T), 'H_abs')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_THICK,   thick,   0_C_INT32_T, 1_C_INT32_T), 'thick')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_T,       T,       0_C_INT32_T, 1_C_INT32_T), 'T')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_PHI,     phi,     0_C_INT32_T, 1_C_INT32_T), 'phi')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_S_BU,    S_bu,    0_C_INT32_T, 1_C_INT32_T), 'S_bu')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_PSI_S,   psi_s,   0_C_INT32_T, 1_C_INT32_T), 'psi_s')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_PSI_L,   psi_l,   0_C_INT32_T, 1_C_INT32_T), 'psi_l')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_PSI_G,   psi_g,   0_C_INT32_T, 1_C_INT32_T), 'psi_g')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_RAY,     ray,     0_C_INT32_T, 1_C_INT32_T), 'ray')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_PERM,    perm,    0_C_INT32_T, 1_C_INT32_T), 'perm')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_FLUSH_V, flush_v, 0_C_INT32_T, 1_C_INT32_T), 'flush_v')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_FLUSH_H, flush_h, 0_C_INT32_T, 1_C_INT32_T), 'flush_h')
    CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_FL_Q,    fl_Q,    0_C_INT32_T, 1_C_INT32_T), 'fl_Q')
    CALL put_sc(h, SC_T_BOTTOM, T_bottom);        CALL put_sc(h, SC_T_TOP, T_top)
    CALL put_sc(h, SC_S_BU_BOTTOM, S_bu_bottom);  CALL put_sc(h, SC_T2M, T2m)
    CALL put_sc(h, SC_FL_Q_BOTTOM, fl_q_bottom)
    CALL put_sc(h, SC_PSI_S_SNOW, psi_s_snow);    CALL put_sc(h, SC_PSI_L_SNOW, psi_l_snow)
    CALL put_sc(h, SC_PSI_G_SNOW, psi_g_snow);    CALL put_sc(h, SC_PHI_S, phi_s)
    CALL put_sc(h, SC_S_ABS_SNOW, S_abs_snow);    CALL put_sc(h, SC_H_ABS_SNOW, H_abs_snow)
    CALL put_sc(h, SC_M_SNOW, m_snow);            CALL put_sc(h, SC_T_SNOW, T_snow)
    CALL put_sc(h, SC_THICK_SNOW, thick_snow);    CALL put_sc(h, SC_LIQUID_PRECIP, liquid_precip)
    CALL put_sc(h, SC_SOLID_PRECIP, solid_precip); CALL put_sc(h, SC_FL_Q_SNOW, fl_q_snow)
    CALL put_sc(h, SC_ALBEDO, albedo);            CALL put_sc(h, SC_FL_SW, fl_sw)
    CALL put_sc(h, SC_FL_LW, fl_lw);              CALL put_sc(h, SC_FL_REST, fl_rest)
    CALL put_sc(h, SC_GRAV_DRAIN, grav_drain);    CALL put_sc(h, SC_GRAV_SALT, grav_salt)
    CALL put_sc(h, SC_GRAV_TEMP, grav_temp);      CALL put_sc(h, SC_MELT_THICK, melt_thick)
    CALL put_sc(h, SC_MELT_THICK_SNOW, melt_thick_snow)
    CALL put_sc(h, SC_MTO1, melt_thick_output(1)); CALL put_sc(h, SC_MTO2, melt_thick_output(2))
    CALL put_sc(h, SC_MTO3, melt_thick_output(3)); CALL put_sc(h, SC_FREEBOARD, freeboard)
    CALL put_sc(h, SC_T_FREEZE, T_freeze);        CALL put_sc(h, SC_MELT_ERR, melt_err)
    CALL put_sc(h, SC_S_TOTAL, S_total)
    CALL put_sc(h, SC_TTOP_WARM, -5._C_DOUBLE)    ! literals of sub_test1 / sub_test4: identity values
    CALL put_sc(h, SC_TTOP_COLD, -10._C_DOUBLE)
    CALL put_sc(h, SC_OFLUX_AMP, 7._C_DOUBLE)
    IF (bgc_flag == 2) THEN                       ! passive tracers: bgc_abs(:,k) is a contiguous column
       CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_BGC_ABS1, bgc_abs(:,1), 0_C_INT32_T, 1_C_INT32_T), 'bgc_abs(:,1)')
       CALL put_sc(h, SC_BGC_BOTTOM1, bgc_bottom(1));  CALL put_sc(h, SC_BGC_TOTAL1, bgc_total(1))
       IF (N_bgc >= 2) THEN
          CALL b200_check(samsim_b200_set_array(h, SAMSIM_ARR_BGC_ABS2, bgc_abs(:,2), 0_C_INT32_T, 1_C_INT32_T), 'bgc_abs(:,2)')
          CALL put_sc(h, SC_BGC_BOTTOM2, bgc_bottom(2));  CALL put_sc(h, SC_BGC_TOTAL2, bgc_total(2))
       END IF
    END IF
    ibuf(1) = N_active
    CALL b200_check(samsim_b200_set_int(h, SAMSIM_INT_N_ACTIVE, ibuf, 0_C_INT32_T, 1_C_INT32_T), 'N_active')
    ibuf(1) = styropor_flag
    CALL b200_check(samsim_b200_set_int(h, SAMSIM_INT_STYROPOR_FLAG, ibuf, 0_C_INT32_T, 1_C_INT32_T), 'styropor_flag')
    CALL b200_check(samsim_b200_set_clock(h, time, INT(i - 1, C_INT64_T), n_time_out, MAX(time_counter, 1)), 'clock')
  END SUBROUTINE b200_push_mo_data

  !> device column 0 -> mo_data (after the loop, or before output()).  If the column hit a reference STOP the
  !! same code is raised here, so the program behaves like the serial model.
  SUBROUTINE b200_pull_mo_data(h)
    USE mo_data
    TYPE(C_PTR), INTENT(in) :: h
    INTEGER(C_INT32_T) :: ibuf(1)
    INTEGER(C_INT64_T) :: i64
    CALL b200_check(samsim_b200_synchronize(h), 'sync')
    CALL b200_check(samsim_b200_get_status(h, ibuf, 0_C_INT32_T, 1_C_INT32_T), 'status')
    IF (ibuf(1) /= 0) THEN
       PRINT*, 'column 1 stopped with the reference STOP code', ibuf(1)
       STOP 1
    END IF
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_M,       m,       0_C_INT32_T, 1_C_INT32_T), 'm')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_S_ABS,   S_abs,   0_C_INT32_T, 1_C_INT32_T), 'S_abs')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_H_ABS,   H_abs,   0_C_INT32_T, 1_C_INT32_T), 'H_abs')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_THICK,   thick,   0_C_INT32_T, 1_C_INT32_T), 'thick')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_T,       T,       0_C_INT32_T, 1_C_INT32_T), 'T')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_PHI,     phi,     0_C_INT32_T, 1_C_INT32_T), 'phi')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_S_BU,    S_bu,    0_C_INT32_T, 1_C_INT32_T), 'S_bu')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_PSI_S,   psi_s,   0_C_INT32_T, 1_C_INT32_T), 'psi_s')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_PSI_L,   psi_l,   0_C_INT32_T, 1_C_INT32_T), 'psi_l')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_PSI_G,   psi_g,   0_C_INT32_T, 1_C_INT32_T), 'psi_g')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_RAY,     ray,     0_C_INT32_T, 1_C_INT32_T), 'ray')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_PERM,    perm,    0_C_INT32_T, 1_C_INT32_T), 'perm')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_FLUSH_V, flush_v, 0_C_INT32_T, 1_C_INT32_T), 'flush_v')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_FLUSH_H, flush_h, 0_C_INT32_T, 1_C_INT32_T), 'flush_h')
    CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_FL_Q,    fl_Q,    0_C_INT32_T, 1_C_INT32_T), 'fl_Q')
    CALL get_sc(h, SC_T_BOTTOM, T_bottom);        CALL get_sc(h, SC_T_TOP, T_top)
    CALL get_sc(h, SC_S_BU_BOTTOM, S_bu_bottom);  CALL get_sc(h, SC_T2M, T2m)
    CALL get_sc(h, SC_FL_Q_BOTTOM, fl_q_bottom)
    CALL get_sc(h, SC_PSI_S_SNOW, psi_s_snow);    CALL get_sc(h, SC_PSI_L_SNOW, psi_l_snow)
    CALL get_sc(h, SC_PSI_G_SNOW, psi_g_snow);    CALL get_sc(h, SC_PHI_S, phi_s)
    CALL get_sc(h, SC_S_ABS_SNOW, S_abs_snow);    CALL get_sc(h, SC_H_ABS_SNOW, H_abs_snow)
    CALL get_sc(h, SC_M_SNOW, m_snow);            CALL get_sc(h, SC_T_SNOW, T_snow)
    CALL get_sc(h, SC_THICK_SNOW, thick_snow);    CALL get_sc(h, SC_LIQUID_PRECIP, liquid_precip)
    CALL get_sc(h, SC_SOLID_PRECIP, solid_precip); CALL get_sc(h, SC_FL_Q_SNOW, fl_q_snow)
    CALL get_sc(h, SC_ENERGY_STORED, energy_stored); CALL get_sc(h, SC_TOTAL_RESIST, total_resist)
    CALL get_sc(h, SC_FRESHWATER, freshwater);    CALL get_sc(h, SC_THICKNESS, thickness)
    CALL get_sc(h, SC_BULK_SALIN, bulk_salin)
    CALL get_sc(h, SC_ALBEDO, albedo);            CALL get_sc(h, SC_FL_SW, fl_sw)
    CALL get_sc(h, SC_FL_LW, fl_lw);              CALL get_sc(h, SC_FL_REST, fl_rest)
    CALL get_sc(h, SC_GRAV_DRAIN, grav_drain);    CALL get_sc(h, SC_GRAV_SALT, grav_salt)
    CALL get_sc(h, SC_GRAV_TEMP, grav_temp);      CALL get_sc(h, SC_MELT_THICK, melt_thick)
    CALL get_sc(h, SC_MELT_THICK_SNOW, melt_thick_snow)
    CALL get_sc(h, SC_MTO1, melt_thick_output(1)); CALL get_sc(h, SC_MTO2, melt_thick_output(2))
    CALL get_sc(h, SC_MTO3, melt_thick_output(3)); CALL get_sc(h, SC_FREEBOARD, freeboard)
    CALL get_sc(h, SC_T_FREEZE, T_freeze);        CALL get_sc(h, SC_MELT_ERR, melt_err)
    IF (bgc_flag == 2) THEN
       CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_BGC_ABS1, bgc_abs(:,1), 0_C_INT32_T, 1_C_INT32_T), 'bgc_abs(:,1)')
       CALL get_sc(h, SC_BGC_BOTTOM1, bgc_bottom(1))
       IF (N_bgc >= 2) THEN
          CALL b200_check(samsim_b200_get_array(h, SAMSIM_ARR_BGC_ABS2, bgc_abs(:,2), 0_C_INT32_T, 1_C_INT32_T), 'bgc_abs(:,2)')
          CALL get_sc(h, SC_BGC_BOTTOM2, bgc_bottom(2))
       END IF
    END IF
    CALL b200_check(samsim_b200_get_int(h, SAMSIM_INT_N_ACTIVE, ibuf, 0_C_INT32_T, 1_C_INT32_T), 'N_active')
    N_active = ibuf(1)
    CALL b200_check(samsim_b200_get_int(h, SAMSIM_INT_STYROPOR_FLAG, ibuf, 0_C_INT32_T, 1_C_INT32_T), 'styropor_flag')
    styropor_flag = ibuf(1)
    CALL b200_check(samsim_b200_get_clock(h, time, i64, n_time_out, time_counter), 'clock')
  END SUBROUTINE b200_pull_mo_data

END MODULE mo_samsim_b200
