"""The inverse-permeability bound of gravity drainage (dm_perm_inv_lo, samsim_b200/csrc/detmath.h) compiled for the
host: below 1/perm with perm = 1e-17*det_pow(1000|psi_l|, 3.10) everywhere, and within 2*DM_PERM_SLACK of it wherever
1/perm is a normal double.  grav_drain's bound pass rules layers out with it (DESIGN §5.1), so a value above 1/perm
could hide a draining layer."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
SRC = HERE / "hostbuild" / "perm_bound_on_host.cpp"
LIB = HERE / "hostbuild" / "_build" / "libperm_bound_on_host.so"


@pytest.fixture(scope="module")
def host():
    deps = [SRC, ROOT / "samsim_b200" / "csrc" / "detmath.h"]
    if not (LIB.exists() and all(LIB.stat().st_mtime > d.stat().st_mtime for d in deps)):
        LIB.parent.mkdir(exist_ok=True)
        r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                            "-o", str(LIB), str(SRC)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    L = C.CDLL(str(LIB))
    dp = C.POINTER(C.c_double)
    L.pb_eval.argtypes = [C.c_int64, dp, dp, dp]
    L.pb_slack.restype = C.c_double

    def ev(psi):
        psi = np.ascontiguousarray(psi, dtype=np.float64)
        perm, inv = np.empty_like(psi), np.empty_like(psi)
        L.pb_eval(psi.size, psi.ctypes.data_as(dp), perm.ctypes.data_as(dp), inv.ctypes.data_as(dp))
        return perm, inv

    return ev, L.pb_slack()


def _sweep():
    """4e6 evenly spaced psi_l in [0, 1] and 6,000 random mantissas in every binade below 1, subnormals included"""
    rng = np.random.default_rng(20261022)
    dense = np.linspace(0.0, 1.0, 4_000_001)
    mant = rng.integers(1, 1 << 52, size=(1023, 6000), dtype=np.int64)
    expo = np.arange(1023, dtype=np.int64)[:, None]  # biased exponent: 0 (subnormals) .. 1022 ([0.5, 1))
    binades = ((expo << 52) | mant).view(np.float64).ravel()
    return np.concatenate([dense, binades, -binades[::1000]])


def test_bound_is_below_inverse_permeability_and_tight(host):
    ev, slack = host
    assert slack == 2.0 ** -16
    psi = _sweep()
    assert psi.size >= 10_000_000
    perm, inv = ev(psi)
    pos = perm > 0.0
    assert np.isfinite(perm).all() and np.isfinite(inv[psi != 0.0]).all()
    # inv * perm in 64-bit-mantissa arithmetic: an error of 2^-63 against a margin of DM_PERM_SLACK/4
    prod = inv[pos].astype(np.longdouble) * perm[pos].astype(np.longdouble)
    assert (prod <= 1.0 - slack / 4).all(), float(prod.max())
    # where 1/perm is normal and the polynomials are used (1000|psi_l| in [2^-256, 2^256]): tight to 2*slack
    x = 1000.0 * np.abs(psi)
    tight = pos & (x >= 2.0 ** -256) & (perm > 1.0 / np.finfo(np.float64).max)
    pt = inv[tight].astype(np.longdouble) * perm[tight].astype(np.longdouble)
    assert (pt >= 1.0 - 2 * slack).all(), float(pt.min())
    # the slack is at least 10x the error of the approximation itself, measured against det_pow
    err = float(np.abs(pt / (1.0 - np.longdouble(slack)) - 1.0).max())
    assert err <= slack / 10, err
    # the layers of a column: psi_l of the bench's mid-winter profile lies in [1e-3, 0.3]
    mid = tight & (np.abs(psi) >= 1e-3) & (np.abs(psi) <= 0.3)
    assert mid.sum() > 1_000_000


def test_bound_at_the_ends(host):
    ev, _ = host
    special = np.array([0.0, -0.0, 1.0, -1.0, np.nan, np.inf, -np.inf, 5e-324, 2.0 ** -270, 1e300, -1e300])
    perm, inv = ev(special)
    assert inv[0] == np.inf and inv[1] == np.inf  # 1/perm with perm = 0
    assert 0.0 < inv[2] * perm[2] < 1.0 and inv[3] == inv[2]
    assert np.isnan(inv[4:7]).all()  # non-finite psi_l: the layer goes to the exact evaluation
    # 1000|psi_l| < 2^-256: the constant 2^790, below 1/perm (perm underflows to 0 or is tiny there)
    assert inv[7] == 2.0 ** 790 and inv[8] == 2.0 ** 790
    assert perm[7] == 0.0 and float(np.longdouble(inv[8]) * np.longdouble(perm[8])) < 1e-2
    assert inv[9] == 0.0 and inv[10] == 0.0  # perm overflows to inf: 1/perm = 0


def test_bound_is_even_in_psi(host):
    ev, _ = host
    psi = np.random.default_rng(7).uniform(0.0, 1.0, 100_000)
    assert np.array_equal(ev(psi)[1], ev(-psi)[1])
