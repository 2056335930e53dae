"""Stochastic forcing without a GPU: the rules of samsim_b200/csrc/noise.cuh compiled for the host against Random123's
known answers, the numpy reference (tests/stochastic_ref.py) and the statistics the contract promises, and the cursor
rule of the window kernel against the pure function."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
sys.path.insert(0, str(HERE))
import stochastic_ref as ref  # noqa: E402

SRC = HERE / "hostbuild" / "noise_on_host.cpp"
LIB = HERE / "hostbuild" / "_build" / "libnoise_on_host.so"

KAT = [  # counter, key -> Philox4x32-10 output (Random123 kat_vectors)
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


def build_lib():
    deps = [SRC, ROOT / "samsim_b200" / "csrc" / "noise.cuh", ROOT / "samsim_b200" / "csrc" / "detmath.h"]
    if not (LIB.exists() and all(LIB.stat().st_mtime > d.stat().st_mtime for d in deps)):
        LIB.parent.mkdir(exist_ok=True)
        r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                            "-o", str(LIB), str(SRC)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    L = C.CDLL(str(LIB))
    dp, ip, up = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint32)
    L.nh_philox.argtypes = [up, up, up]
    for f in (L.nh_det_log, L.nh_det_cos, L.nh_det_exp):
        f.argtypes = [C.c_int64, dp, dp]
    L.nh_normals.argtypes = [C.c_uint64, C.c_int32, C.c_int32, ip, C.c_int32, C.c_int32, dp]
    L.nh_series.argtypes = [C.c_uint64, C.c_double, C.c_double, C.c_int32, C.c_int32, ip, C.c_int32, C.c_int32, dp]
    L.nh_window.restype = C.c_int32
    L.nh_window.argtypes = [C.c_uint64, C.c_double, C.c_double, C.c_int32, C.c_int32, ip, C.c_int32, C.c_int32,
                            C.c_int32, dp, dp]
    L.nh_apply.argtypes = [C.c_int32, C.c_double, C.c_double, C.c_int64, dp, dp, dp]
    return L


class Host:
    """numpy-facing wrappers of the host build"""

    def __init__(self, L):
        self.L = L

    def _vec(self, f, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty_like(x)
        f(x.size, _p(x, C.c_double), _p(out, C.c_double))
        return out

    def det_log(self, x):
        return self._vec(self.L.nh_det_log, x)

    def det_cos(self, x):
        return self._vec(self.L.nh_det_cos, x)

    def det_exp(self, x):
        return self._vec(self.L.nh_det_exp, x)

    def philox(self, ctr, key):
        c, k = np.array(ctr, dtype=np.uint32), np.array(key, dtype=np.uint32)
        out = np.empty(4, dtype=np.uint32)
        self.L.nh_philox(_p(c, C.c_uint32), _p(k, C.c_uint32), _p(out, C.c_uint32))
        return out

    def normals(self, seed, kind, streams, rec0, nrec):
        s = np.ascontiguousarray(streams, dtype=np.int32)
        out = np.empty((len(s), nrec))
        self.L.nh_normals(seed, kind, len(s), _p(s, C.c_int32), rec0, nrec, _p(out, C.c_double))
        return out

    def series(self, seed, sigma, phi, kind, streams, rec0, nrec):
        s = np.ascontiguousarray(streams, dtype=np.int32)
        out = np.empty((len(s), nrec))
        self.L.nh_series(seed, sigma, phi, kind, len(s), _p(s, C.c_int32), rec0, nrec, _p(out, C.c_double))
        return out

    def window(self, seed, sigma, phi, kind, streams, cursor, first, last, state):
        s = np.ascontiguousarray(streams, dtype=np.int32)
        out = np.empty((len(s), last - first + 1))
        cur = self.L.nh_window(seed, sigma, phi, kind, len(s), _p(s, C.c_int32), cursor, first, last,
                               _p(state, C.c_double), _p(out, C.c_double))
        return cur, out

    def apply(self, mode, sigma, v, e):
        v, e = np.ascontiguousarray(v, dtype=np.float64), np.ascontiguousarray(e, dtype=np.float64)
        out = np.empty_like(v)
        self.L.nh_apply(mode, sigma, 0.5, v.size, _p(v, C.c_double), _p(e, C.c_double), _p(out, C.c_double))
        return out


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


@pytest.fixture(scope="module")
def host():
    return Host(build_lib())


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(host, ctr, key, want):
    assert host.philox(ctr, key).tolist() == list(want)
    assert ref.philox(np.array(ctr), np.array(key)).tolist() == list(want)


def test_philox_matches_numpy_over_many_counters_and_keys(host):
    rng = np.random.default_rng(1)
    ctr = rng.integers(0, 2 ** 32, (2000, 4), dtype=np.uint64)
    key = rng.integers(0, 2 ** 32, (2000, 2), dtype=np.uint64)
    ctr[:10] = 0
    ctr[10:20, 0] = 2 ** 32 - 1
    key[20:30] = 2 ** 32 - 1
    want = ref.philox(ctr, key)
    got = np.stack([host.philox(c, k) for c, k in zip(ctr, key)])
    assert np.array_equal(got, want)


def test_uniform_is_inside_the_open_interval():
    assert ref.uniform(0, 0) == 0.5 * 2.0 ** -52
    assert ref.uniform(0xFFFFFFFF, 0xFFFFFFFF) == 1.0 - 0.5 * 2.0 ** -52


@pytest.mark.parametrize("seed", [0, 12345, 0xDEADBEEF12345678])
def test_normals_match_numpy(host, seed):
    streams = np.array([0, 1, 7, 4095, 1_048_575, 2 ** 31 - 1])
    for kind in range(4):
        want = ref.normals(seed, kind, streams, np.arange(1, 301), host.det_log, host.det_cos)
        assert np.array_equal(bits(host.normals(seed, kind, streams, 1, 300)), bits(want))


@pytest.mark.parametrize("seed,sigma,phi", [(3, 2.5, 0.9), (0xFFFFFFFFFFFFFFFF, 0.3, 0.0), (2 ** 40 + 17, 1.0, 0.99)])
def test_series_matches_numpy_bit_for_bit(host, seed, sigma, phi):
    streams = np.array([0, 5, 6, 1000, 123_456])
    for kind in range(4):
        want = ref.series(seed, sigma, phi, kind, streams, 3000, host.det_log, host.det_cos)
        got = host.series(seed, sigma, phi, kind, streams, 1, 3000)
        assert np.array_equal(bits(got), bits(want)), kind
        # a later start gives the same values: the function of the record
        assert np.array_equal(bits(host.series(seed, sigma, phi, kind, streams, 1777, 40)), bits(want[:, 1776:1816]))


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_modes_match_numpy(host, mode):
    rng = np.random.default_rng(mode)
    sigma = 0.7
    v = rng.normal(size=5000) * 300.0
    v[:5] = [0.0, -0.0, 1.0, -1.0, 250.0]
    e = rng.normal(size=5000) * sigma
    e[5:8] = [-1.0, -3.0, 0.0]
    want = ref.apply(mode, sigma, v, e, host.det_exp)
    assert np.array_equal(bits(host.apply(mode, sigma, v, e)), bits(want))


def test_statistics(host):
    """1,000 streams x 1,200 records per kind: mean 0, variance sigma^2, lag-1 autocorrelation phi, no correlation
    between streams or kinds; lognormal keeps the mean.  Tolerances: about four standard errors."""
    seed, sigma, phi, nstr, nrec = 99, 1.7, 0.8, 1000, 1200
    streams = np.arange(nstr)
    e = np.stack([host.series(seed, sigma, phi, k, streams, 1, nrec) for k in range(4)])   # [4, nstr, nrec]
    n = nstr * nrec
    # AR(1): the effective number of independent samples of a stream is nrec * (1 - phi) / (1 + phi)
    n_eff = nstr * nrec * (1 - phi) / (1 + phi)
    for k in range(4):
        x = e[k]
        assert abs(x.mean()) < 4 * sigma / np.sqrt(n_eff), k
        assert abs(x.var() / sigma ** 2 - 1) < 4 * np.sqrt(2 / n_eff), k
        r1 = (x[:, 1:] * x[:, :-1]).mean() / x.var()
        assert abs(r1 - phi) < 4 * np.sqrt((1 - phi ** 2) / n), k
        # neighbouring streams, and stream s against stream s + 500
        for a, b in ((x[:-1], x[1:]), (x[:500], x[500:])):
            rho = (a * b).mean() / np.sqrt((a * a).mean() * (b * b).mean())
            assert abs(rho) < 4 * np.sqrt((1 + phi ** 2) / (1 - phi ** 2) / a.size), k
    for k, j in ((0, 1), (1, 2), (2, 3), (0, 3)):
        rho = (e[k] * e[j]).mean() / np.sqrt((e[k] ** 2).mean() * (e[j] ** 2).mean())
        assert abs(rho) < 4 * np.sqrt((1 + phi ** 2) / (1 - phi ** 2) / n), (k, j)
    # white noise (phi = 0): the normals themselves
    z = host.series(seed, 1.0, 0.0, 2, streams, 1, nrec)
    assert abs(z.mean()) < 4 / np.sqrt(n) and abs(z.var() - 1) < 4 * np.sqrt(2 / n)
    # lognormal: E[exp(e - sigma^2 / 2)] = 1, whose variance is exp(sigma^2) - 1
    s_ln = 0.3
    eln = host.series(seed, s_ln, phi, 3, streams, 1, nrec)
    m = host.apply(2, s_ln, np.ones(eln.size), eln.ravel())
    n_eff_ln = n * (1 - phi * np.exp(s_ln ** 2 * phi)) / (1 + phi)   # rough, lag correlations of exp(e) are larger
    assert abs(m.mean() - 1) < 4 * np.sqrt((np.exp(s_ln ** 2) - 1) / max(n_eff_ln, n_eff / 4))


def test_cursor_rule_gives_the_pure_function(host):
    """launch windows of random lengths (up to 24 records, overlapping by one like the step's), with backward and
    forward jumps of the clock, replayed through the window rule with held state: every window equals the pure
    function of the record"""
    rng = np.random.default_rng(4)
    seed, sigma, phi = 2024, 3.0, 0.95
    streams = np.array([0, 3, 3, 77, 4096])
    nrec = 700
    pure = host.series(seed, sigma, phi, 1, streams, 1, nrec)
    state = np.zeros(2 * len(streams))
    cursor, tc = 0, 1
    restarts = jumps = 0
    for _ in range(400):
        u = rng.random()
        if u < 0.05:
            tc = int(rng.integers(1, tc + 1))          # set_clock back, or a checkpoint of an earlier time
            jumps += 1
        elif u < 0.08:
            tc = min(nrec - 30, tc + int(rng.integers(2, 40)))   # set_clock forward
        first = max(tc - 1, 1)
        last = min(first + int(rng.integers(0, 24)), nrec)
        restarts += not (cursor >= 1 and first >= cursor - 1)
        new, e = host.window(seed, sigma, phi, 1, streams, cursor, first, last, state)
        assert np.array_equal(bits(e), bits(pure[:, first - 1:last])), (cursor, first, last)
        assert new == (cursor if cursor >= 1 and first >= cursor - 1 and cursor > last else last)
        cursor = new
        # the held values are e(cursor-1) and e(cursor)
        assert np.array_equal(bits(state[1::2]), bits(pure[:, cursor - 1]))
        if cursor > 1:
            assert np.array_equal(bits(state[0::2]), bits(pure[:, cursor - 2]))
        tc = last if last < nrec - 30 else 1
    assert restarts > 5 and jumps > 5
