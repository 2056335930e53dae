"""Time statistics without a GPU: the rules of samsim_b200/csrc/time_stats.cuh compiled for the host against the numpy
reference (tests/time_stats_ref.py), and the window count of a call against a step-by-step replay of the clock."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
sys.path.insert(0, str(HERE))
from time_stats_ref import Acc  # noqa: E402

SRC = HERE / "hostbuild" / "time_stats_on_host.cpp"
LIB = HERE / "hostbuild" / "_build" / "libtime_stats_on_host.so"


@pytest.fixture(scope="module")
def lib():
    deps = [SRC, ROOT / "samsim_b200" / "csrc" / "time_stats.cuh", ROOT / "samsim_b200" / "csrc" / "group_stats.cuh"]
    if not (LIB.exists() and all(LIB.stat().st_mtime > d.stat().st_mtime for d in deps)):
        LIB.parent.mkdir(exist_ok=True)
        r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                            "-o", str(LIB), str(SRC)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    L = C.CDLL(str(LIB))
    dp = C.POINTER(C.c_double)
    L.tsh_accumulate.argtypes = [C.c_int32, C.c_int32, dp, C.POINTER(C.c_uint8), dp]
    L.tsh_records_in.restype = C.c_int64
    L.tsh_records_in.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_int64]
    L.tsh_windows_completed.restype = C.c_int64
    L.tsh_windows_completed.argtypes = [C.c_int32, C.c_int64, C.c_int64]
    return L


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def host(L, x, c):
    x, c = np.ascontiguousarray(x, dtype=np.float64), np.ascontiguousarray(c, dtype=np.uint8)
    out = np.empty((x.shape[1], 5))
    L.tsh_accumulate(x.shape[0], x.shape[1], _p(x, C.c_double), _p(c, C.c_uint8), _p(out, C.c_double))
    return out


def numpy_ref(x, c):
    a = Acc(x.shape[1])
    for r in range(x.shape[0]):
        a.update(x[r], c[r].astype(bool))
    return a.finish()


def test_accumulate_matches_numpy(lib):
    rng = np.random.default_rng(7)
    nrec, nq = 40, 300
    x = rng.normal(size=(nrec, nq)) * 10.0 ** rng.integers(-6, 6, (1, nq))
    x[:, :20] += 1e6                                    # large offsets: the recurrence's rounding matters
    c = rng.random((nrec, nq)) < 0.7
    c[:, 0] = False                                     # n = 0
    c[:, 1] = False
    c[13, 1] = True                                     # n = 1
    assert np.array_equal(bits(host(lib, x, c)), bits(numpy_ref(x, c)))


def test_count_zero_and_one(lib):
    x = np.array([[-0.0, 3.5, 2.0], [7.0, -1.25, 9.0]])
    c = np.array([[True, True, False], [False, False, False]])
    out = host(lib, x, c)
    assert np.array_equal(bits(out), bits(numpy_ref(x, c)))
    assert out[0, 0] == 1 and not np.signbit(out[0, 1]) and out[0, 2] == 0.0   # mean = 0 + (-0.0) / 1 = +0.0
    assert np.signbit(out[0, 3]) and np.signbit(out[0, 4])                    # min and max keep -0.0
    assert out[1].tolist()[:3] == [1.0, 3.5, 0.0]
    assert out[2, 0] == 0 and np.isnan(out[2, 1:]).all()


@pytest.mark.parametrize("first", [0.0, -0.0])
def test_signed_zero_ties_keep_the_earlier_value(lib, first):
    x = np.array([[first], [-first], [first], [-first]])
    c = np.ones_like(x, dtype=bool)
    out = host(lib, x, c)
    assert np.array_equal(bits(out), bits(numpy_ref(x, c)))
    assert np.signbit(out[0, 3]) == np.signbit(first) and np.signbit(out[0, 4]) == np.signbit(first)
    # a smaller value replaces the zero, a NaN accumulator takes the first value
    x2 = np.array([[0.0], [-1.0], [0.5]])
    out2 = host(lib, x2, np.ones_like(x2, dtype=bool))
    assert out2[0, 3] == -1.0 and out2[0, 4] == 0.5
    assert np.array_equal(bits(out2), bits(numpy_ref(x2, np.ones_like(x2, dtype=bool))))


def _replay(i, n_time_out, i_time_out, nsteps):
    """loop indices of the records that nsteps steps write, by the clock of samsim_b200_step"""
    recs = []
    for _ in range(nsteps):
        i += 1
        out = n_time_out == i_time_out or i == 1
        n_time_out = 0 if out else n_time_out + 1
        if out:
            recs.append(i)
    return recs


@pytest.mark.parametrize("i_time_out", [0, 1, 4, 99])
def test_records_in_matches_the_clock(lib, i_time_out):
    for i, nto in [(0, 0), (0, i_time_out), (1, 0), (17, min(3, i_time_out)), (500, i_time_out)]:
        for nsteps in [0, 1, 2, 5, i_time_out, i_time_out + 1, i_time_out + 2, 3 * i_time_out + 7, 1000]:
            assert lib.tsh_records_in(i, nto, i_time_out, nsteps) == len(_replay(i, nto, i_time_out, nsteps)), \
                (i, nto, nsteps)


@pytest.mark.parametrize("rpw", [0, 1, 3, 7])
def test_windows_completed_by_a_call(lib, rpw):
    """window boundaries counted record by record against the rule, for calls from the first record (i = 0 -> 1) on"""
    i_time_out = 4
    for in_window0 in range(max(rpw, 1)):
        for nsteps in range(0, 60):
            nrec = lib.tsh_records_in(0, 0, i_time_out, nsteps)
            recs = _replay(0, 0, i_time_out, nsteps)
            assert nrec == len(recs) and (not recs or recs[0] == 1)
            cur, done = in_window0, 0
            for _ in recs:
                cur += 1
                if rpw > 0 and cur == rpw:
                    done, cur = done + 1, 0
            assert lib.tsh_windows_completed(rpw, in_window0, nrec) == done, (in_window0, nsteps)
