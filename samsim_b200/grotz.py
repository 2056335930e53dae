"""Python face of the C++ host layer (include/samsim_b200_host.h): grotz(testcase, description) for batches.

`grotz()` is the batched mirror of the reference's entry point (mo_grotz.f90:83): it initialises the testcase,
reads the forcing files, runs the time loop on the GPU and writes dat_*.dat in the reference's formats.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from . import api


class _HostCase(C.Structure):
    _fields_ = [("cfg", api._CConfig), ("N_active", C.c_int32), ("i_time", C.c_int32), ("time_total", C.c_double),
                ("arrays", C.POINTER(C.c_double) * len(api.ARRAY_IDS)), ("scalars", C.c_double * len(api.SCALAR_IDS)),
                ("length_input_lab", C.c_int64)]


class _GrotzOptions(C.Structure):
    _fields_ = [("ncol", C.c_int32), ("device", C.c_int32), ("forcing_dir", C.c_char_p), ("output_dir", C.c_char_p),
                ("max_steps", C.c_int64), ("forcing_scale", C.POINTER(C.c_double)), ("forcing_offset", C.POINTER(C.c_double)),
                ("ttop_warm", C.POINTER(C.c_double)), ("ttop_cold", C.POINTER(C.c_double)), ("oflux_amp", C.POINTER(C.c_double)),
                ("quiet", C.c_int32), ("lab_input_dir", C.c_char_p)]


class _GrotzMember(C.Structure):
    _fields_ = [("testcase", C.c_int32), ("description", C.c_char_p), ("output_dir", C.c_char_p), ("max_steps", C.c_int64)]


def _lib():
    L = api.load_library()
    L.samsim_host_init_testcase.restype = C.c_int
    L.samsim_host_init_testcase.argtypes = [C.c_int32, C.POINTER(_HostCase)]
    L.samsim_host_case_free.argtypes = [C.POINTER(_HostCase)]
    L.samsim_host_read_forcing.restype = C.c_int
    L.samsim_host_read_forcing.argtypes = [C.c_char_p, C.c_int32, C.POINTER(C.c_double)]
    L.samsim_host_read_lab_series.restype = C.c_int
    L.samsim_host_read_lab_series.argtypes = [C.c_char_p, C.c_int32, C.c_int64, C.POINTER(C.c_double)]
    L.samsim_grotz.restype = C.c_int
    L.samsim_grotz.argtypes = [C.c_int32, C.c_char_p, C.POINTER(_GrotzOptions)]
    L.samsim_grotz_batch.restype = C.c_int
    L.samsim_grotz_batch.argtypes = [C.POINTER(_GrotzMember), C.c_int32, C.POINTER(_GrotzOptions), C.POINTER(C.c_int32)]
    return L


def init_testcase(testcase: int) -> dict:
    """mo_init.f90's init(testcase) as a dict keyed by mo_data names (host only, no GPU needed)."""
    L = _lib()
    hc = _HostCase()
    rc = L.samsim_host_init_testcase(testcase, C.byref(hc))
    if rc != 0:
        raise api.SamsimError(rc, f"testcase {testcase} is not covered (1-9, 33, 34, 50, 99, 101-105, 111)")
    try:
        N = hc.cfg.Nlayer
        st = {n: getattr(hc.cfg, n) for n in api._CFG_INT_FIELDS + api._CFG_DBL_FIELDS}
        for name, a in api.ARRAY_IDS.items():
            ext = N - 1 if name == "ray" else (N + 1 if name == "fl_Q" else N)
            st[name] = np.ctypeslib.as_array(hc.arrays[a], shape=(ext,)).copy()
        for name, q in api.SCALAR_IDS.items():
            st[name] = hc.scalars[q]
        st.update(N_active=hc.N_active, i_time=hc.i_time, time_total=hc.time_total, length_input_lab=hc.length_input_lab,
                  status=0, styropor_flag=0, time=0.0, i=0, n_time_out=0, time_counter=1)
        return st
    finally:
        L.samsim_host_case_free(C.byref(hc))


def read_forcing(directory, nrec: int = 13148) -> np.ndarray:
    L = _lib()
    out = np.empty((4, nrec))
    rc = L.samsim_host_read_forcing(str(directory).encode(), nrec, api._dp(out))
    if rc != 0:
        raise api.SamsimError(rc, f"cannot read the four *.txt.input files in {directory}")
    return out


def read_lab_series(directory, testcase: int, nrec: int) -> np.ndarray:
    """mo_grotz.f90:138-169: {Tice,snowfall,heat,styropor}_exp_<testcase-100>.txt -> [4, nrec]"""
    L = _lib()
    out = np.empty((4, nrec))
    rc = L.samsim_host_read_lab_series(str(directory).encode(), testcase, nrec, api._dp(out))
    if rc != 0:
        raise api.SamsimError(rc, f"cannot read {nrec} records of the four lab series of testcase {testcase} in {directory}")
    return out


def grotz(testcase: int, description: str = "", *, output_dir, forcing_dir=".", ncol: int = 1, device: int = 0,
          max_steps: int = 0, forcing_scale=None, forcing_offset=None, ttop_warm=None, ttop_cold=None, oflux_amp=None,
          quiet: bool = True, lab_input_dir="2017_input") -> int:
    """Run grotz(testcase, description) on the GPU; returns 0 or the reference STOP code of column 0."""
    L = _lib()
    Path(output_dir).mkdir(parents=True, exist_ok=True)
    keep = []

    def vec(a, shape):
        if a is None:
            return None
        v = np.ascontiguousarray(a, dtype=np.float64).reshape(shape)
        keep.append(v)
        return api._dp(v)
    o = _GrotzOptions(ncol=ncol, device=device, forcing_dir=str(forcing_dir).encode(), output_dir=str(output_dir).encode(),
                      max_steps=max_steps, forcing_scale=vec(forcing_scale, (4, ncol)), forcing_offset=vec(forcing_offset, (4, ncol)),
                      ttop_warm=vec(ttop_warm, (ncol,)), ttop_cold=vec(ttop_cold, (ncol,)), oflux_amp=vec(oflux_amp, (ncol,)),
                      quiet=int(quiet), lab_input_dir=str(lab_input_dir).encode())
    rc = L.samsim_grotz(testcase, description.encode(), C.byref(o))
    if rc < 0:
        raise api.SamsimError(rc, L.samsim_b200_last_error().decode())
    return rc


def grotz_batch(members, *, device: int = 0, forcing_dir=None, lab_input_dir=None, quiet: bool = True) -> list[int]:
    """Run several grotz(testcase, description) at once, one GPU column each, every member to its own end.

    `members`: dicts with `testcase`, `output_dir` and optionally `description` and `max_steps` (0 = i_time).  The
    testcases must share one configuration; 101-105 may be mixed.  Each member writes the dat_*.dat files grotz()
    writes for it alone.  Returns each member's code: 0 or its reference STOP code.  forcing_dir / lab_input_dir
    None = the reference's defaults ("." and "2017_input").
    """
    L = _lib()
    ms = (_GrotzMember * len(members))() if members else None
    for q, m in enumerate(members):
        Path(m["output_dir"]).mkdir(parents=True, exist_ok=True)
        ms[q] = _GrotzMember(testcase=int(m["testcase"]), description=str(m.get("description", "")).encode(),
                             output_dir=str(m["output_dir"]).encode(), max_steps=int(m.get("max_steps", 0)))
    o = _GrotzOptions(ncol=0, device=device, forcing_dir=None if forcing_dir is None else str(forcing_dir).encode(),
                      output_dir=None, max_steps=0, quiet=int(quiet),
                      lab_input_dir=None if lab_input_dir is None else str(lab_input_dir).encode())
    codes = (C.c_int32 * max(len(members), 1))()
    rc = L.samsim_grotz_batch(ms, len(members), C.byref(o), codes)
    if rc < 0:
        why = {-1: "bad argument (members, or an option that belongs to samsim_grotz)",
               -4: "the members' testcases do not share one configuration"}
        raise api.SamsimError(rc, why.get(rc) or L.samsim_b200_last_error().decode())
    return [int(c) for c in codes[:len(members)]]
