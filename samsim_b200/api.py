"""ctypes binding of include/samsim_b200.h.

Plumbing only: all physics runs in the CUDA library.  If the library is missing or no GPU is
present the constructors raise -- there is deliberately no CPU path here.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field, fields
from pathlib import Path

import numpy as np

import os

_ROOT = Path(__file__).resolve().parent
# SAMSIM_B200_LIB selects another build of the SAME library (tuning variants under samsim_b200/_lib/)
_LIB_PATH = Path(os.environ.get("SAMSIM_B200_LIB", _ROOT / "_lib" / "libsamsim_b200.so"))


class SamsimError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"samsim_b200 error {code}: {msg}")
        self.code = code


def lib_path() -> Path:
    return _LIB_PATH


# ---- ids: must mirror include/samsim_b200.h ---------------------------------------------------
ARRAY_IDS = {n: i for i, n in enumerate(
    ["m", "S_abs", "H_abs", "thick", "T", "phi", "S_bu", "psi_s", "psi_l", "psi_g", "ray", "perm", "flush_v",
     "flush_h", "fl_Q", "bgc_abs1", "bgc_abs2"])}
SCALAR_IDS = {n: i for i, n in enumerate(
    ["T_bottom", "T_top", "S_bu_bottom", "T2m", "fl_q_bottom", "psi_s_snow", "psi_l_snow", "psi_g_snow", "phi_s",
     "S_abs_snow", "H_abs_snow", "m_snow", "T_snow", "thick_snow", "liquid_precip", "solid_precip", "fl_q_snow",
     "energy_stored", "total_resist", "freshwater", "thickness", "bulk_salin", "albedo", "fl_sw", "fl_lw", "fl_rest",
     "grav_drain", "grav_salt", "grav_temp", "melt_thick", "melt_thick_snow", "melt_thick_snow_old",
     "melt_thick_output1", "melt_thick_output2", "melt_thick_output3", "freeboard", "T_freeze", "melt_err", "S_total",
     "ttop_warm", "ttop_cold", "oflux_amp", "bgc_bottom1", "bgc_bottom2", "bgc_total1", "bgc_total2"])}
INT_IDS = {"N_active": 0, "status": 1, "styropor_flag": 2, "events0": 3, "events1": 4}
# branch events, order of samsim_event_id (include/samsim_b200.h): bit id of events0 (id < 32) / events1 (id - 32)
EVENT_NAMES = [
    "flood", "flood_neg_free", "flood_simple", "flush3", "flush4", "flush_inline", "styropor", "snow_thermo",
    "snow_thermo_meltwater", "snow_wet", "snow_merge", "snow_compaction", "snow_coupling_iter", "snow_coupling_warm1",
    "snow_coupling_warm2", "snow_precip", "snow_precip_0", "melt_snow_all", "melt_snow_part", "bottom_melt",
    "bottom_melt_simple_a", "bottom_melt_simple_b", "bottom_growth_simple", "bottom_growth", "top_grow_a", "top_grow_b",
    "top_grow_c", "top_melt_a", "top_melt_b", "top_melt_c", "grav_drained", "salt_clamp",
    "gas_refill", "getT_Tfr_fallback", "getT_saltfree", "getT_liquid", "heat_melt", "heat_thin_snow", "melt_thick_gas",
    "snow_meltwater_to_ice", "prescribe", "grav_drain_simple", "notzflux", "flush3_clamp", "scrub", "melt_thick", "turb",
    "tank", "two_pass_step"]


def decode_events(ev0: int, ev1: int) -> set:
    """names of the branch events whose bits are set in the two event words of a column"""
    w = (int(ev0) & 0xFFFFFFFF) | ((int(ev1) & 0xFFFFFFFF) << 32)
    return {n for j, n in enumerate(EVENT_NAMES) if (w >> j) & 1}
SNAP_SCALARS = ["freeboard", "thick_snow", "T_snow", "psi_l_snow", "psi_s_snow", "energy_stored", "freshwater",
                "total_resist", "thickness", "bulk_salin", "grav_drain", "grav_salt", "grav_temp", "T2m", "T_top",
                "melt_thick_output1", "melt_thick_output2", "melt_thick_output3", "time", "N_active"]
SNAP_ARRAYS = ["T", "psi_s", "thick", "S_bu", "ray", "psi_l", "perm", "flush_v", "flush_h", "psi_g",
               "bgc1_bu", "bgc1_br", "bgc2_bu", "bgc2_br"]
SNAP_NONE, SNAP_SCALARS_ONLY, SNAP_FULL = 0, 1, 2

_CFG_INT_FIELDS = ["testcase", "Nlayer", "N_top", "N_middle", "N_bottom", "atmoflux_flag", "grav_flag",
                   "prescribe_flag", "grav_heat_flag", "flush_heat_flag", "turb_flag", "salt_flag", "boundflux_flag",
                   "flush_flag", "flood_flag", "bottom_flag", "precip_flag", "harmonic_flag", "tank_flag",
                   "albedo_flag", "lab_snow_flag", "freeboard_snow_flag", "snow_flush_flag", "snow_precip_flag",
                   "i_time_out", "N_bgc"]
_CFG_DBL_FIELDS = ["dt", "thick_0", "thick_min", "time_out", "alpha_flux_instable", "alpha_flux_stable", "m_total",
                   "max_flux_plate", "k_snow_flush", "k_styropor"]


class _CConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in _CFG_INT_FIELDS] + [(n, C.c_double) for n in _CFG_DBL_FIELDS]


@dataclass
class Config:
    """samsim_config_t: flags of mo_data.f90:136-155 with the defaults of mo_init.f90:83-109."""
    testcase: int = 0
    Nlayer: int = 0
    N_top: int = 0
    N_middle: int = 0
    N_bottom: int = 0
    atmoflux_flag: int = 1
    grav_flag: int = 2
    prescribe_flag: int = 1
    grav_heat_flag: int = 1
    flush_heat_flag: int = 1
    turb_flag: int = 2
    salt_flag: int = 1
    boundflux_flag: int = 1
    flush_flag: int = 5
    flood_flag: int = 2
    bottom_flag: int = 1
    precip_flag: int = 0
    harmonic_flag: int = 2
    tank_flag: int = 1
    albedo_flag: int = 2
    lab_snow_flag: int = 0
    freeboard_snow_flag: int = 0
    snow_flush_flag: int = 1
    snow_precip_flag: int = 1
    i_time_out: int = 0
    N_bgc: int = 0  # passive tracers: 0 = bgc_flag 1; 1..2 = bgc_flag 2 with that many tracers
    dt: float = 0.0
    thick_0: float = 0.0
    thick_min: float = 0.0
    time_out: float = 0.0
    alpha_flux_instable: float = 0.0
    alpha_flux_stable: float = 0.0
    m_total: float = 0.0
    max_flux_plate: float = 10000.0
    k_snow_flush: float = 0.75
    k_styropor: float = 0.8

    def to_c(self) -> _CConfig:
        c = _CConfig()
        for f in fields(self):
            setattr(c, f.name, getattr(self, f.name))
        return c

    @classmethod
    def from_state(cls, st: dict) -> "Config":
        """Build from a dict keyed by mo_data names (e.g. an oracle state)."""
        kw = {}
        for f in fields(cls):
            if f.name in st:
                kw[f.name] = type(f.default)(st[f.name])
        if "bgc_flag" in st:  # mo_data carries bgc_flag and N_bgc; the C config only N_bgc (0 = no tracers)
            kw["N_bgc"] = int(st.get("N_bgc", 0)) if int(st["bgc_flag"]) == 2 else 0
        return cls(**kw)


_lib = None


def load_library() -> C.CDLL:
    """dlopen the in-tree CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise SamsimError(-3, f"{_LIB_PATH} is missing: run `python -m samsim_b200.build` (nvcc, sm_100a). "
                              "samsim_b200 has no CPU fallback.")
    L = C.CDLL(str(_LIB_PATH))
    H = C.c_void_p
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    sig = {
        "samsim_b200_create": (C.c_int, [C.POINTER(_CConfig), C.c_int32, C.c_int32, C.POINTER(H)]),
        "samsim_b200_destroy": (None, [H]),
        "samsim_b200_last_error": (C.c_char_p, []),
        "samsim_b200_version": (C.c_char_p, []),
        "samsim_b200_array_extent": (C.c_int32, [H, C.c_int32]),
        "samsim_b200_set_array": (C.c_int, [H, C.c_int32, dp, C.c_int32, C.c_int32]),
        "samsim_b200_get_array": (C.c_int, [H, C.c_int32, dp, C.c_int32, C.c_int32]),
        "samsim_b200_set_scalar": (C.c_int, [H, C.c_int32, dp, C.c_int32, C.c_int32]),
        "samsim_b200_get_scalar": (C.c_int, [H, C.c_int32, dp, C.c_int32, C.c_int32]),
        "samsim_b200_set_int": (C.c_int, [H, C.c_int32, ip, C.c_int32, C.c_int32]),
        "samsim_b200_get_int": (C.c_int, [H, C.c_int32, ip, C.c_int32, C.c_int32]),
        "samsim_b200_broadcast_column": (C.c_int, [H, C.c_int32, C.c_int32, C.c_int32]),
        "samsim_b200_set_clock": (C.c_int, [H, C.c_double, C.c_int64, C.c_int32, C.c_int32]),
        "samsim_b200_get_clock": (C.c_int, [H, dp, C.POINTER(C.c_int64), ip, ip]),
        "samsim_b200_set_forcing": (C.c_int, [H, C.c_int32, C.c_int32, dp, ip, dp, dp]),
        "samsim_b200_update_forcing": (C.c_int, [H, dp]),
        "samsim_b200_update_forcing_records": (C.c_int, [H, C.c_int32, C.c_int32, dp]),
        "samsim_b200_set_lab_forcing": (C.c_int, [H, C.c_int32, C.c_int64, dp, ip]),
        "samsim_b200_set_lab_lengths": (C.c_int, [H, C.c_int32, C.POINTER(C.c_int64)]),
        "samsim_b200_step": (C.c_int, [H, C.c_int64]),
        "samsim_b200_set_end_step": (C.c_int, [H, C.POINTER(C.c_int64), C.c_int32, C.c_int32]),
        "samsim_b200_synchronize": (C.c_int, [H]),
        "samsim_b200_steps_to_next_output": (C.c_int64, [H]),
        "samsim_b200_set_snapshot_mode": (C.c_int, [H, C.c_int32]),
        "samsim_b200_get_snapshot": (C.c_int, [H, dp, dp, C.c_int32, C.c_int32]),
        "samsim_b200_set_group_stats": (C.c_int, [H, C.c_int32, ip, C.c_int32, dp, C.c_uint32, C.c_int32]),
        "samsim_b200_group_stats_held": (C.c_int32, [H]),
        "samsim_b200_get_group_stats": (C.c_int, [H, dp, dp, C.POINTER(C.c_int64), C.c_int32, C.c_int32]),
        "samsim_b200_clear_group_stats": (C.c_int, [H]),
        "samsim_b200_set_time_stats": (C.c_int, [H, C.c_int32, C.c_uint32, C.c_int32, dp, C.c_uint32, C.c_int32]),
        "samsim_b200_time_stats_held": (C.c_int32, [H]),
        "samsim_b200_get_time_stats": (C.c_int, [H, dp, ip, dp, C.POINTER(C.c_int64), C.c_int32, C.c_int32, C.c_int32,
                                                 C.c_int32]),
        "samsim_b200_close_time_window": (C.c_int, [H]),
        "samsim_b200_clear_time_stats": (C.c_int, [H]),
        "samsim_b200_get_status": (C.c_int, [H, ip, C.c_int32, C.c_int32]),
        "samsim_b200_count_failed": (C.c_int, [H, ip]),
        "samsim_b200_reduce_diag": (C.c_int, [H, dp]),
        "samsim_b200_launch_count": (C.c_int64, [H]),
        "samsim_b200_last_step_ms": (C.c_int, [H, C.POINTER(C.c_float)]),
        "samsim_b200_device_layout": (C.c_int, [H, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                                C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
        "samsim_b200_save_checkpoint": (C.c_int, [H, C.c_char_p]),
        "samsim_b200_load_checkpoint": (C.c_int, [H, C.c_char_p]),
        "samsim_b200_rebin": (C.c_int, [H, ip]),
        "samsim_b200_set_tuning": (C.c_int, [H, C.c_int32, C.c_int32]),
        "samsim_b200_set_rebin_interval": (C.c_int, [H, C.c_int64]),
        "samsim_b200_set_rebin_auto": (C.c_int, [H, C.c_double]),
        "samsim_b200_get_divergence": (C.c_int, [H, dp, dp, C.POINTER(C.c_int64)]),
        "samsim_b200_get_slot_map": (C.c_int, [H, ip]),
        "samsim_b200_kat_getT": (C.c_int, [C.c_int32, C.c_int32, dp, dp, dp, dp, dp, ip, C.c_int32]),
        "samsim_b200_kat_scalar": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, dp, dp, dp, C.c_int32]),
        "samsim_b200_fp64_peak": (C.c_int, [C.c_int32, C.c_double, dp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "samsim_b200_create", "samsim_b200_destroy", "samsim_b200_last_error", "samsim_b200_version",
    "samsim_b200_array_extent", "samsim_b200_set_array", "samsim_b200_get_array", "samsim_b200_set_scalar",
    "samsim_b200_get_scalar", "samsim_b200_set_int", "samsim_b200_get_int", "samsim_b200_broadcast_column",
    "samsim_b200_set_clock", "samsim_b200_get_clock", "samsim_b200_set_forcing", "samsim_b200_update_forcing",
    "samsim_b200_update_forcing_records",
    "samsim_b200_set_lab_forcing", "samsim_b200_set_lab_lengths", "samsim_b200_set_end_step",
    "samsim_b200_step", "samsim_b200_synchronize", "samsim_b200_steps_to_next_output",
    "samsim_b200_set_snapshot_mode", "samsim_b200_get_snapshot", "samsim_b200_set_group_stats",
    "samsim_b200_group_stats_held", "samsim_b200_get_group_stats", "samsim_b200_clear_group_stats",
    "samsim_b200_set_time_stats", "samsim_b200_time_stats_held", "samsim_b200_get_time_stats",
    "samsim_b200_close_time_window", "samsim_b200_clear_time_stats",
    "samsim_b200_get_status",
    "samsim_b200_count_failed", "samsim_b200_reduce_diag", "samsim_b200_launch_count", "samsim_b200_last_step_ms",
    "samsim_b200_device_layout", "samsim_b200_save_checkpoint", "samsim_b200_load_checkpoint", "samsim_b200_rebin", "samsim_b200_set_tuning", "samsim_b200_set_rebin_interval", "samsim_b200_set_rebin_auto", "samsim_b200_get_divergence", "samsim_b200_get_slot_map",
    "samsim_b200_kat_getT", "samsim_b200_kat_scalar", "samsim_b200_fp64_peak",
]


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32)) if a is not None else None


def _lp(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64)) if a is not None else None


def _check(L, rc):
    if rc != 0:
        raise SamsimError(rc, L.samsim_b200_last_error().decode())


class Engine:
    """A batch of `ncol` independent columns resident on one GPU."""

    def __init__(self, cfg: Config, ncol: int, device: int = 0):
        self.L = load_library()
        self.cfg = cfg
        self.ncol = int(ncol)
        self.device = device
        self.h = C.c_void_p()
        cc = cfg.to_c()
        _check(self.L, self.L.samsim_b200_create(C.byref(cc), self.ncol, device, C.byref(self.h)))

    def close(self):
        if getattr(self, "h", None):
            self.L.samsim_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- state ------------------------------------------------------------------------------
    def extent(self, name: str) -> int:
        return self.L.samsim_b200_array_extent(self.h, ARRAY_IDS[name])

    def set_array(self, name: str, values, col0: int = 0):
        v = np.ascontiguousarray(values, dtype=np.float64)
        ext = self.extent(name)
        v = v.reshape(-1, ext)
        _check(self.L, self.L.samsim_b200_set_array(self.h, ARRAY_IDS[name], _dp(v), col0, v.shape[0]))

    def get_array(self, name: str, col0: int = 0, n: int | None = None) -> np.ndarray:
        n = self.ncol - col0 if n is None else n
        out = np.empty((n, self.extent(name)), dtype=np.float64)
        _check(self.L, self.L.samsim_b200_get_array(self.h, ARRAY_IDS[name], _dp(out), col0, n))
        return out

    def set_scalar(self, name: str, values, col0: int = 0):
        v = np.ascontiguousarray(np.atleast_1d(values), dtype=np.float64)
        _check(self.L, self.L.samsim_b200_set_scalar(self.h, SCALAR_IDS[name], _dp(v), col0, v.shape[0]))

    def get_scalar(self, name: str, col0: int = 0, n: int | None = None, out: np.ndarray | None = None) -> np.ndarray:
        n = self.ncol - col0 if n is None else n
        out = np.empty(n, dtype=np.float64) if out is None else out
        assert out.shape == (n,) and out.dtype == np.float64 and out.flags.c_contiguous
        _check(self.L, self.L.samsim_b200_get_scalar(self.h, SCALAR_IDS[name], _dp(out), col0, n))
        return out

    def set_int(self, name: str, values, col0: int = 0):
        v = np.ascontiguousarray(np.atleast_1d(values), dtype=np.int32)
        _check(self.L, self.L.samsim_b200_set_int(self.h, INT_IDS[name], _ip(v), col0, v.shape[0]))

    def get_int(self, name: str, col0: int = 0, n: int | None = None) -> np.ndarray:
        n = self.ncol - col0 if n is None else n
        out = np.empty(n, dtype=np.int32)
        _check(self.L, self.L.samsim_b200_get_int(self.h, INT_IDS[name], _ip(out), col0, n))
        return out

    def events(self, col: int = 0) -> set:
        """branch events column `col` has executed since the event words were last cleared (names of EVENT_NAMES)"""
        return decode_events(self.get_int("events0", col, 1)[0], self.get_int("events1", col, 1)[0])

    def clear_events(self):
        z = np.zeros(self.ncol, dtype=np.int32)
        self.set_int("events0", z)
        self.set_int("events1", z)

    def broadcast_column(self, src: int = 0, col0: int = 0, n: int | None = None):
        n = self.ncol - col0 if n is None else n
        _check(self.L, self.L.samsim_b200_broadcast_column(self.h, src, col0, n))

    def set_clock(self, time: float, i: int, n_time_out: int, time_counter: int = 1):
        _check(self.L, self.L.samsim_b200_set_clock(self.h, float(time), int(i), int(n_time_out), int(time_counter)))

    def get_clock(self) -> dict:
        t, i, n, tc = C.c_double(), C.c_int64(), C.c_int32(), C.c_int32()
        _check(self.L, self.L.samsim_b200_get_clock(self.h, C.byref(t), C.byref(i), C.byref(n), C.byref(tc)))
        return {"time": t.value, "i": i.value, "n_time_out": n.value, "time_counter": tc.value}

    def load_column_state(self, st: dict, col: int = 0, set_clock: bool = True):
        """Load one column from a dict keyed by mo_data names (arrays 0-based, Fortran element 1 first)."""
        for name in ARRAY_IDS:
            if name in st and self.extent(name) > 0:  # tracer arrays exist only with N_bgc > 0
                self.set_array(name, np.asarray(st[name], dtype=np.float64)[None, :self.extent(name)], col0=col)
        for name in SCALAR_IDS:
            if name in st:
                self.set_scalar(name, [st[name]], col0=col)
        for name in INT_IDS:
            if name in st:
                self.set_int(name, [st[name]], col0=col)
        if set_clock:
            self.set_clock(st["time"], st["i"], st["n_time_out"], max(int(st.get("time_counter", 1)), 1))

    def column_state(self, col: int = 0) -> dict:
        d = {n: self.get_array(n, col, 1)[0] for n in ARRAY_IDS if self.extent(n) > 0}
        d.update({n: float(self.get_scalar(n, col, 1)[0]) for n in SCALAR_IDS})
        d.update({n: int(self.get_int(n, col, 1)[0]) for n in INT_IDS})
        d.update(self.get_clock())
        return d

    # ---- forcing ----------------------------------------------------------------------------
    def set_forcing(self, series, site_of_col=None, scale=None, offset=None):
        """series[nsite, 4, nrec] in kind order fl_sw, fl_lw, T2m, precip; site_of_col[ncol]; scale/offset[4, ncol].
        Any nsite is accepted, up to one series per column or more (a grid cell per column, a time-shifted series
        per ensemble member); only device memory limits the table."""
        s = np.ascontiguousarray(series, dtype=np.float64)
        if s.ndim == 2:
            s = s[None]
        nsite, four, nrec = s.shape
        assert four == 4
        soc = None if site_of_col is None else np.ascontiguousarray(site_of_col, dtype=np.int32)
        sc = None if scale is None else np.ascontiguousarray(scale, dtype=np.float64).reshape(4, self.ncol)
        of = None if offset is None else np.ascontiguousarray(offset, dtype=np.float64).reshape(4, self.ncol)
        _check(self.L, self.L.samsim_b200_set_forcing(self.h, nsite, nrec, _dp(s), _ip(soc), _dp(sc), _dp(of)))

    def update_forcing(self, series):
        """Refresh the base series in place (same shape as the last set_forcing); `series` may be a pinned buffer."""
        s = series if isinstance(series, np.ndarray) and series.flags.c_contiguous and series.dtype == np.float64 \
            else np.ascontiguousarray(series, dtype=np.float64)
        _check(self.L, self.L.samsim_b200_update_forcing(self.h, _dp(s)))

    def update_forcing_records(self, rec0: int, series):
        """Refresh records rec0 .. rec0+n-1 (1-based) of every site and kind from series[nsite, 4, n]; the other
        records of the table are kept."""
        s = np.ascontiguousarray(series, dtype=np.float64)
        if s.ndim == 2:
            s = s[None]
        assert s.ndim == 3 and s.shape[1] == 4
        _check(self.L, self.L.samsim_b200_update_forcing_records(self.h, int(rec0), s.shape[2], _dp(s)))

    def set_lab_forcing(self, series, set_of_col=None, nrec_of_set=None):
        """series[nset, 4, nrec] in kind order Tice, snowfall, heat, styropor.  nrec_of_set[nset]: the real length of
        each set when the sets are padded to a common nrec (None = every set holds nrec records)."""
        s = np.ascontiguousarray(series, dtype=np.float64)
        if s.ndim == 2:
            s = s[None]
        nset, four, nrec = s.shape
        assert four == 4
        soc = None if set_of_col is None else np.ascontiguousarray(set_of_col, dtype=np.int32)
        _check(self.L, self.L.samsim_b200_set_lab_forcing(self.h, nset, nrec, _dp(s), _ip(soc)))
        if nrec_of_set is not None:
            ln = np.ascontiguousarray(nrec_of_set, dtype=np.int64)
            assert ln.shape == (nset,)
            _check(self.L, self.L.samsim_b200_set_lab_lengths(self.h, nset, _lp(ln)))

    def set_end_step(self, values, col0: int = 0):
        """Last loop index i each of the columns col0, col0+1, ... runs; past it the column is frozen with status 0
        (INT64_MAX = no end, the default)."""
        v = np.ascontiguousarray(np.atleast_1d(values), dtype=np.int64)
        _check(self.L, self.L.samsim_b200_set_end_step(self.h, _lp(v), col0, v.shape[0]))

    # ---- stepping ---------------------------------------------------------------------------
    def step(self, nsteps: int = 1, sync: bool = True):
        _check(self.L, self.L.samsim_b200_step(self.h, int(nsteps)))
        if sync:
            self.synchronize()

    def synchronize(self):
        _check(self.L, self.L.samsim_b200_synchronize(self.h))

    def steps_to_next_output(self) -> int:
        return int(self.L.samsim_b200_steps_to_next_output(self.h))

    def set_snapshot_mode(self, mode: int):
        _check(self.L, self.L.samsim_b200_set_snapshot_mode(self.h, mode))

    def get_snapshot(self, col0: int = 0, n: int | None = None, arrays: bool = True, out_scalars: np.ndarray | None = None):
        """S8 record of columns [col0, col0+n).  `out_scalars` (n x 20, C-contiguous float64, e.g. a pinned buffer)
        receives the scalars without an allocation."""
        n = self.ncol - col0 if n is None else n
        sc = out_scalars if out_scalars is not None else np.empty((n, len(SNAP_SCALARS)), dtype=np.float64)
        assert sc.shape == (n, len(SNAP_SCALARS)) and sc.flags.c_contiguous and sc.dtype == np.float64
        ar = np.empty((n, len(SNAP_ARRAYS), self.cfg.Nlayer), dtype=np.float64) if arrays else None
        _check(self.L, self.L.samsim_b200_get_snapshot(self.h, _dp(sc), _dp(ar), col0, n))
        out = {name: sc[:, j] for j, name in enumerate(SNAP_SCALARS)}
        if arrays:
            for j, name in enumerate(SNAP_ARRAYS):
                out[name] = ar[:, j, : (self.cfg.Nlayer - 1 if name == "ray" else self.cfg.Nlayer)]
        return out

    # ---- group statistics at S8 records -------------------------------------------------------
    def set_group_stats(self, group_of_col=None, depths=(), profiles=(), max_records: int = 64, ngroup: int | None = None):
        """Ensemble statistics per column group at every output record, kept on the device (include/samsim_b200.h).
        group_of_col[ncol] in [-1, ngroup), -1 = in no group, None = one group of every column; ngroup defaults to
        max(group_of_col) + 1, and 0 switches the statistics off.  depths: metres below the ice surface; profiles:
        names of SNAP_ARRAYS.  Needs snapshot mode SCALARS, FULL with profiles."""
        goc = None if group_of_col is None else np.ascontiguousarray(group_of_col, dtype=np.int32)
        if ngroup is None:
            ngroup = 1 if goc is None else int(goc.max()) + 1
        assert goc is None or goc.shape == (self.ncol,)
        z = np.ascontiguousarray(depths, dtype=np.float64).reshape(-1)
        mask = 0
        for name in profiles:
            mask |= 1 << SNAP_ARRAYS.index(name)
        _check(self.L, self.L.samsim_b200_set_group_stats(self.h, int(ngroup), _ip(goc), len(z), _dp(z) if len(z) else None,
                                                          mask, int(max_records)))
        self._gs = {"ngroup": int(ngroup), "depths": z.copy(),
                    "profiles": [n for j, n in enumerate(SNAP_ARRAYS) if mask >> j & 1]} if ngroup else None

    def group_stats_held(self) -> int:
        return int(self.L.samsim_b200_group_stats_held(self.h))

    def group_stats(self, clear: bool = True, rec0: int = 0, nrec: int | None = None) -> dict:
        """The held records: time[R], i[R], quantities [(name, depth or None)] and count / mean / var / min / max of
        shape [R, G, Q].  clear=True drops the held records afterwards."""
        g = getattr(self, "_gs", None)
        assert g is not None, "group statistics are off"
        nrec = self.group_stats_held() - rec0 if nrec is None else nrec
        qn = [(n, None) for n in SNAP_SCALARS] + [(p, float(d)) for p in g["profiles"] for d in g["depths"]]
        st = np.empty((nrec, g["ngroup"], len(qn), 5), dtype=np.float64)
        t = np.empty(nrec, dtype=np.float64)
        i = np.empty(nrec, dtype=np.int64)
        _check(self.L, self.L.samsim_b200_get_group_stats(self.h, _dp(st), _dp(t), _lp(i), int(rec0), int(nrec)))
        if clear:
            _check(self.L, self.L.samsim_b200_clear_group_stats(self.h))
        out = {"time": t, "i": i, "quantities": qn}
        for k, name in enumerate(("count", "mean", "var", "min", "max")):
            out[name] = st[..., k]
        return out

    def clear_group_stats(self):
        _check(self.L, self.L.samsim_b200_clear_group_stats(self.h))

    # ---- time statistics over windows of S8 records -------------------------------------------
    def set_time_stats(self, records_per_window: int, scalars=None, depths=(), profiles=(), max_windows: int = 64):
        """Per-column count, mean, variance, min and max over windows of output records, accumulated on the device
        (include/samsim_b200.h).  A window collects records_per_window records; 0 = windows end only at
        close_time_window().  scalars: names of SNAP_SCALARS (None = all 20); depths: metres below the ice surface;
        profiles: names of SNAP_ARRAYS.  No scalars and no profiles switch the statistics off.  Needs snapshot mode
        SCALARS, FULL with profiles.  A new setting drops the held windows and the window in progress."""
        sc = list(SNAP_SCALARS) if scalars is None else list(scalars)
        scmask = 0
        for name in sc:
            scmask |= 1 << SNAP_SCALARS.index(name)
        z = np.ascontiguousarray(depths, dtype=np.float64).reshape(-1)
        mask = 0
        for name in profiles:
            mask |= 1 << SNAP_ARRAYS.index(name)
        _check(self.L, self.L.samsim_b200_set_time_stats(self.h, int(records_per_window), scmask, len(z),
                                                         _dp(z) if len(z) else None, mask, int(max_windows)))
        qn = [(n, None) for j, n in enumerate(SNAP_SCALARS) if scmask >> j & 1]
        qn += [(p, float(d)) for j, p in enumerate(SNAP_ARRAYS) if mask >> j & 1 for d in z]
        self._ts = {"quantities": qn} if qn else None

    def time_stats_held(self) -> int:
        return int(self.L.samsim_b200_time_stats_held(self.h))

    def time_stats(self, col0: int = 0, n: int | None = None, clear: bool = False) -> dict:
        """The held windows for caller columns col0..col0+n-1: nrec, time_first, time_last, i_first, i_last of shape
        [W]; quantities [(name, depth or None)]; count / mean / var / min / max of shape [W, n, Q].  clear=True drops
        the held windows afterwards."""
        t = getattr(self, "_ts", None)
        assert t is not None, "time statistics are off"
        n = self.ncol - col0 if n is None else n
        W, qn = self.time_stats_held(), t["quantities"]
        st = np.empty((W, n, len(qn), 5), dtype=np.float64)
        nrec = np.empty(W, dtype=np.int32)
        tm = np.empty((W, 2), dtype=np.float64)
        i = np.empty((W, 2), dtype=np.int64)
        _check(self.L, self.L.samsim_b200_get_time_stats(self.h, _dp(st), _ip(nrec), _dp(tm), _lp(i), 0, W, int(col0), int(n)))
        if clear:
            self.clear_time_stats()
        out = {"nrec": nrec, "time_first": tm[:, 0], "time_last": tm[:, 1], "i_first": i[:, 0], "i_last": i[:, 1],
               "quantities": qn}
        for k, name in enumerate(("count", "mean", "var", "min", "max")):
            out[name] = st[..., k]
        return out

    def close_time_window(self):
        _check(self.L, self.L.samsim_b200_close_time_window(self.h))

    def clear_time_stats(self):
        _check(self.L, self.L.samsim_b200_clear_time_stats(self.h))

    # ---- diagnostics ------------------------------------------------------------------------
    def status(self) -> np.ndarray:
        return self.get_int("status")

    def count_failed(self) -> int:
        v = C.c_int32()
        _check(self.L, self.L.samsim_b200_count_failed(self.h, C.byref(v)))
        return v.value

    def save_checkpoint(self, path) -> None:
        _check(self.L, self.L.samsim_b200_save_checkpoint(self.h, str(path).encode()))

    def load_checkpoint(self, path) -> None:
        _check(self.L, self.L.samsim_b200_load_checkpoint(self.h, str(path).encode()))

    def rebin(self) -> bool:
        """Sort the columns by regime on the device (SURVEY 8e); column numbering seen by the caller is unchanged."""
        v = C.c_int32()
        _check(self.L, self.L.samsim_b200_rebin(self.h, C.byref(v)))
        return bool(v.value)

    def set_tuning(self, two_pass: bool, prefetch_layers: int = 0) -> None:
        """kernel tuning (results do not depend on it): merged forward / backward passes for steady columns; L1
        prefetch distance of the layer sweeps (0 = keep the default)"""
        _check(self.L, self.L.samsim_b200_set_tuning(self.h, int(bool(two_pass)), int(prefetch_layers)))

    def set_rebin_interval(self, nsteps: int) -> None:
        _check(self.L, self.L.samsim_b200_set_rebin_interval(self.h, int(nsteps)))

    def set_rebin_auto(self, idle_share_threshold: float) -> None:
        """re-bin whenever the kernel-measured share of idle lane-layers of the last launch exceeds the threshold"""
        _check(self.L, self.L.samsim_b200_set_rebin_auto(self.h, float(idle_share_threshold)))

    def divergence(self) -> dict:
        """warp divergence of the last launch, measured in the kernel (reductions / ballots per warp)"""
        a, b, n = C.c_double(), C.c_double(), C.c_int64()
        _check(self.L, self.L.samsim_b200_get_divergence(self.h, C.byref(a), C.byref(b), C.byref(n)))
        return {"idle_lane_layer_share": a.value, "snow_class_split_warp_share": b.value, "rebins": n.value}

    def slot_map(self) -> np.ndarray:
        out = np.empty(self.ncol, dtype=np.int32)
        _check(self.L, self.L.samsim_b200_get_slot_map(self.h, out.ctypes.data_as(C.POINTER(C.c_int32))))
        return out

    def reduce_diag(self) -> dict:
        out = np.empty(18, dtype=np.float64)
        _check(self.L, self.L.samsim_b200_reduce_diag(self.h, _dp(out)))
        names = ["thickness", "bulk_salin", "freeboard", "thick_snow", "T_top", "N_active"]
        return {n: {"sum": out[3 * j], "min": out[3 * j + 1], "max": out[3 * j + 2]} for j, n in enumerate(names)}

    def launch_count(self) -> int:
        return int(self.L.samsim_b200_launch_count(self.h))

    def last_step_ms(self) -> float:
        v = C.c_float()
        _check(self.L, self.L.samsim_b200_last_step_ms(self.h, C.byref(v)))
        return v.value


# ---- unit KAT entry points ---------------------------------------------------------------------
def kat_getT(salt_flag: int, H, S_bu, T_in, device: int = 0):
    L = load_library()
    H, S_bu, T_in = (np.ascontiguousarray(x, dtype=np.float64) for x in (H, S_bu, T_in))
    n = len(H)
    T, phi, st = np.empty(n), np.empty(n), np.empty(n, dtype=np.int32)
    _check(L, L.samsim_b200_kat_getT(salt_flag, n, _dp(H), _dp(S_bu), _dp(T_in), _dp(T), _dp(phi), _ip(st), device))
    # low 16 bits: STOP code; above: the getT branch bits of event word 1 (bit SAMSIM_EV_GETT_* - 32)
    return T, phi, st & 0xFFFF, (st >> 16) & 0xFFFF


def kat_scalar(fn: int, salt_flag: int, a, b=None, device: int = 0):
    L = load_library()
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
    out = np.empty(len(a))
    _check(L, L.samsim_b200_kat_scalar(fn, salt_flag, len(a), _dp(a), _dp(b), _dp(out), device))
    return out


def fp64_peak(device: int = 0, seconds: float = 1.0) -> float:
    L = load_library()
    v = C.c_double()
    _check(L, L.samsim_b200_fp64_peak(device, seconds, C.byref(v)))
    return v.value
