"""Correlated stochastic forcing without a GPU: the rules of samsim_b200/csrc/noise.cuh (the argument rules, the Cholesky
factor, the four-kind basis window and the column mix) compiled for the host against the numpy reference
(tests/correlated_ref.py) and the statistics DESIGN §7.4 promises, the cursor rule per basis stream, and the bilinear
basis helper."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from samsim_b200 import api, distributed

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE))
import correlated_ref as cref  # noqa: E402
from test_stochastic_forcing_cpu import Host, build_lib  # noqa: E402

ROOT = HERE.parent
SRC = HERE / "hostbuild" / "correlated_noise_on_host.cpp"
LIB = HERE / "hostbuild" / "_build" / "libcorrelated_noise_on_host.so"

SIGMA = [0.25, 12.0, 1.5, 0.6]
PHI = [0.7, 0.8, 0.9, 0.5]
# cloudier sky: more LW and warmer T2m, less SW; precipitation with the cloud
CORR = np.array([[1.0, -0.6, -0.3, -0.2],
                 [-0.6, 1.0, 0.5, 0.3],
                 [-0.3, 0.5, 1.0, 0.1],
                 [-0.2, 0.3, 0.1, 1.0]])
NEAR_SINGULAR = np.array([[1.0, 0.999999, 0.5, 0.0],
                          [0.999999, 1.0, 0.5, 0.0],
                          [0.5, 0.5, 1.0, -0.25],
                          [0.0, 0.0, -0.25, 1.0]])
EQUICORR = np.full((4, 4), 0.4) + 0.6 * np.eye(4)
MATRICES = {"none": None, "identity": np.eye(4), "cloud": CORR, "near_singular": NEAR_SINGULAR, "equicorr": EQUICORR}

dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)


def build_corr_lib():
    deps = [SRC, ROOT / "samsim_b200" / "csrc" / "noise.cuh", ROOT / "samsim_b200" / "csrc" / "detmath.h"]
    if not (LIB.exists() and all(LIB.stat().st_mtime > d.stat().st_mtime for d in deps)):
        LIB.parent.mkdir(exist_ok=True)
        r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                            "-o", str(LIB), str(SRC)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    L = C.CDLL(str(LIB))
    L.nh_check.restype = C.c_int32
    L.nh_check.argtypes = [dp, dp, ip, dp, C.c_int32, C.c_int64, ip, dp, ip, dp, C.c_char_p]
    L.nh_cholesky.restype = C.c_int32
    L.nh_cholesky.argtypes = [dp, dp]
    L.nh_basis_window.restype = C.c_int32
    L.nh_basis_window.argtypes = [C.c_uint64, dp, dp, dp, C.c_int32, ip, C.c_int32, C.c_int32, C.c_int32, dp, dp]
    L.nh_mix.argtypes = [C.c_int32, C.c_int32, ip, dp, C.c_int32, dp, dp, dp, ip]
    L.nh_apply_mixed.argtypes = [C.c_int32, C.c_double, C.c_int64, dp, dp, dp, dp]
    return L


class CorrHost(Host):
    """numpy-facing wrappers of the correlated host build (tests/hostbuild/correlated_noise_on_host.cpp); the
    single-stream rules and detmath come from the host build of noise_on_host.cpp (Host)"""

    def __init__(self):
        super().__init__(build_lib())
        self.C = build_corr_lib()

    def check(self, sigma, phi, mode, corr, nmix, ncol, basis, weight):
        """None for a valid setting (and then (on, single, L)), else the message"""
        sg, ph = np.ascontiguousarray(sigma, np.float64), np.ascontiguousarray(phi, np.float64)
        md = np.ascontiguousarray(mode, np.int32)
        cr = None if corr is None else np.ascontiguousarray(corr, np.float64).reshape(16)
        b = None if basis is None else np.ascontiguousarray(basis, np.int32).reshape(-1)
        w = None if weight is None else np.ascontiguousarray(weight, np.float64).reshape(-1)
        os_, L = np.zeros(2, np.int32), np.zeros(16)
        msg = C.create_string_buffer(256)
        rc = self.C.nh_check(_p(sg, dp), _p(ph, dp), _p(md, ip), _p(cr, dp), nmix, ncol, _p(b, ip), _p(w, dp),
                             _p(os_, ip), _p(L, dp), msg)
        return msg.value.decode() if rc else (bool(os_[0]), bool(os_[1]), L.reshape(4, 4))

    def cholesky(self, corr):
        c = np.ascontiguousarray(corr, np.float64).reshape(16)
        L = np.zeros(16)
        return L.reshape(4, 4) if self.C.nh_cholesky(_p(c, dp), _p(L, dp)) else None

    def basis_window(self, seed, sigma, phi, corr, ids, cursor, first, last, state=None):
        """(new cursor, E[n, 4, last-first+1]); state[n, 4, 2] updated in place"""
        ids = np.ascontiguousarray(ids, np.int32)
        sg, ph = np.ascontiguousarray(sigma, np.float64), np.ascontiguousarray(phi, np.float64)
        cr = None if corr is None else np.ascontiguousarray(corr, np.float64).reshape(16)
        if state is None:
            state = np.zeros((len(ids), 4, 2))
        out = np.empty((len(ids), 4, last - first + 1))
        cur = self.C.nh_basis_window(seed, _p(sg, dp), _p(ph, dp), _p(cr, dp), len(ids), _p(ids, ip), cursor, first,
                                     last, _p(state, dp), _p(out, dp))
        return cur, out

    def mix(self, idx, weight, E):
        idx = np.ascontiguousarray(idx, np.int32)
        weight = np.ascontiguousarray(weight, np.float64).reshape(idx.shape)
        E = np.ascontiguousarray(E, np.float64)
        ncol, nmix = idx.shape
        e, q, has = np.empty((ncol, E.shape[1])), np.empty(ncol), np.empty(ncol, np.int32)
        self.C.nh_mix(ncol, nmix, _p(idx, ip), _p(weight, dp), E.shape[1], _p(E, dp), _p(e, dp), _p(q, dp), _p(has, ip))
        return e, q, has.astype(bool)

    def apply_mixed(self, mode, sigma, v, e, q):
        v, e, q = (np.ascontiguousarray(np.broadcast_to(x, np.shape(v)), np.float64) for x in (v, e, q))
        out = np.empty_like(v)
        self.C.nh_apply_mixed(mode, sigma, v.size, _p(v, dp), _p(e, dp), _p(q, dp), _p(out, dp))
        return out


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


@pytest.fixture(scope="module")
def host():
    return CorrHost()


# ---- the Cholesky factor --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", [n for n in MATRICES if MATRICES[n] is not None])
def test_cholesky_matches_numpy_bit_for_bit(host, name):
    c = MATRICES[name]
    got, want = host.cholesky(c), cref.cholesky(c)
    assert np.array_equal(bits(got), bits(want))
    assert np.allclose(got @ got.T, c, rtol=0, atol=1e-12)
    assert np.allclose(got, np.linalg.cholesky(c), rtol=0, atol=1e-9)


def test_cholesky_rejects_what_is_not_positive_definite(host):
    singular = np.ones((4, 4))
    indefinite = np.eye(4)
    indefinite[0, 1] = indefinite[1, 0] = 1.2
    for c in (singular, indefinite):
        assert host.cholesky(c) is None and cref.cholesky(c) is None


# ---- the basis window and the mix against numpy ---------------------------------------------------------------------
@pytest.mark.parametrize("name", list(MATRICES))
def test_basis_window_matches_numpy_bit_for_bit(host, name):
    seed, ids = 0xC0FFEE_1234, np.array([0, 1, 7, 4095, 1_048_575, 2 ** 31 - 1])
    sigma = [0.25, 0.0, 1.5, 0.6]   # a sigma-0 kind still draws its normals for the others
    want = cref.basis_series(seed, sigma, PHI, MATRICES[name], ids, 3000, host.det_log, host.det_cos)   # [4, n, r]
    _, got = host.basis_window(seed, sigma, PHI, MATRICES[name], ids, 0, 1, 3000)
    assert np.array_equal(bits(got.transpose(1, 0, 2)), bits(want))
    # a later start is the same function of the record
    _, mid = host.basis_window(seed, sigma, PHI, MATRICES[name], ids, 0, 1777, 1816)
    assert np.array_equal(bits(mid.transpose(1, 0, 2)), bits(want[:, :, 1776:1816]))


def test_identity_basis_window_is_the_single_stream_series(host):
    """corr NULL or the identity: w = z, so each kind's E is the e of samsim_b200_set_stochastic_forcing"""
    seed, ids = 77, np.array([0, 3, 123_456])
    for corr in (None, np.eye(4)):
        _, got = host.basis_window(seed, SIGMA, PHI, corr, ids, 0, 1, 3000)
        for k in range(4):
            assert np.array_equal(bits(got[:, k]), bits(host.series(seed, SIGMA[k], PHI[k], k, ids, 1, 3000))), k


@pytest.mark.parametrize("nmix", range(1, 9))
def test_mix_matches_numpy_bit_for_bit(host, nmix):
    rng = np.random.default_rng(nmix)
    nb, ncol, nrec = 12, 40, 3000
    E = rng.normal(size=(nb, nrec)) * 3.0
    E[:, :3] = [0.0, -0.0, 1e-300]
    idx = np.stack([rng.permutation(nb)[:nmix] for _ in range(ncol)]).astype(np.int32)
    idx[rng.random(idx.shape) < 0.3] = -1     # empty entries
    idx[0] = -1                               # a column with none
    w = rng.normal(size=idx.shape)            # negative weights
    w[1] = 1.0
    e, q, has = host.mix(idx, w, E)
    ids = np.arange(nb)
    e_ref, q_ref, has_ref = cref.mix(idx, w, ids, E)
    assert np.array_equal(has, has_ref) and not has[0]
    assert np.array_equal(bits(e), bits(e_ref)) and np.array_equal(bits(q[has]), bits(q_ref[has]))
    # one entry of weight 1.0 is the basis value itself, -0.0 included
    one = np.full((nb, nmix), -1, np.int32)
    one[:, nmix - 1] = np.arange(nb)
    e1, q1, _ = host.mix(one, np.ones(one.shape), E)
    assert np.array_equal(bits(e1), bits(E)) and (q1 == 1.0).all()


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_modes_with_mixed_weights_match_numpy(host, mode):
    rng = np.random.default_rng(10 + mode)
    sigma = 0.7
    v = rng.normal(size=5000) * 300.0
    v[:5] = [0.0, -0.0, 1.0, -1.0, 250.0]
    e = rng.normal(size=5000) * sigma
    e[5:8] = [-1.0, -3.0, 0.0]
    q = rng.uniform(0.2, 3.0, 5000)
    want = cref.apply(mode, sigma, v, e, q, host.det_exp)
    assert np.array_equal(bits(host.apply_mixed(mode, sigma, v, e, q)), bits(want))
    # q = 1.0 is the single-stream mode
    assert np.array_equal(bits(host.apply_mixed(mode, sigma, v, e, 1.0)), bits(host.apply(mode, sigma, v, e)))


@pytest.mark.parametrize("name", ["none", "cloud", "near_singular"])
def test_perturbed_columns_match_numpy(host, name):
    """the whole chain: basis window, mix and modes, for columns of nmix 5 with empty entries and negative weights"""
    rng = np.random.default_rng(5)
    seed, ncol, nrec, nmix = 31337, 30, 3000, 5
    ids = np.array([2, 9, 40, 41, 1000, 70_000])
    basis = np.stack([rng.permutation(ids)[:nmix] for _ in range(ncol)]).astype(np.int32)
    basis[rng.random(basis.shape) < 0.25] = -1
    basis[3] = -1
    w = rng.normal(size=basis.shape)
    values = rng.uniform(50, 300, (ncol, 4, nrec))
    mode = [1, 0, 0, 2]
    sigma = [0.25, 12.0, 0.0, 0.6]
    want = cref.perturbed(seed, sigma, PHI, mode, MATRICES[name], basis, w, values, host.det_log, host.det_cos,
                          host.det_exp)
    _, E = host.basis_window(seed, sigma, PHI, MATRICES[name], ids, 0, 1, nrec)   # [nb, 4, nrec]
    idx = np.where(basis >= 0, np.searchsorted(ids, basis), -1).astype(np.int32)
    got = values.copy()
    for k in range(4):
        if sigma[k] == 0.0:
            continue
        e, q, has = host.mix(idx, w, E[:, k])
        got[has, k] = host.apply_mixed(mode[k], sigma[k], values[has, k], e[has], np.repeat(q[has, None], nrec, 1))
    assert np.array_equal(bits(got), bits(want))
    assert np.array_equal(bits(want[3]), bits(values[3])) and np.array_equal(bits(want[:, 2]), bits(values[:, 2]))


# ---- statistics -----------------------------------------------------------------------------------------------------
def _moments(host, seed, sigma, phi, corr, nb=10_000, nrec=3000, skip=100, chunk=500):
    """over nb basis streams x records skip+1..nrec: the innovations' and E's lag-0 cross-kind products, E's second
    moments (the first records are left out: from record 1 the cross-covariance of kinds with different phi relaxes
    to its stationary value)"""
    ww, ee, ez = np.zeros((4, 4)), np.zeros((4, 4)), np.zeros(4)
    n = 0
    for b0 in range(0, nb, chunk):
        ids = np.arange(b0, b0 + chunk)
        _, E = host.basis_window(seed, sigma, phi, corr, ids, 0, 1, nrec)
        E = E[:, :, skip:].transpose(1, 0, 2).reshape(4, -1)
        ee += E @ E.T
        ez += E.sum(axis=1)
        n += E.shape[1]
        if b0 == 0:   # the innovations themselves: phi 0, sigma 1
            _, W = host.basis_window(seed, [1.0] * 4, [0.0] * 4, corr, np.arange(nb), 0, 1, 120)
            W = W.transpose(1, 0, 2).reshape(4, -1)
            ww = (W @ W.T) / W.shape[1]
    return ww, ee / n, ez / n, n


def test_statistics_of_correlated_kinds(host):
    """10,000 basis streams x 3,000 records: the innovations correlate by corr, E by the phi formula of DESIGN §7.4.
    Tolerances: four standard errors."""
    seed = 4242
    ww, ee, mean, n = _moments(host, seed, SIGMA, PHI, CORR)
    nw = 10_000 * 120
    for i in range(4):
        assert abs(ww[i, i] - 1.0) < 4 * np.sqrt(2 / nw)
        for j in range(i):
            r = CORR[i, j]
            assert abs(ww[i, j] - r) < 4 * (1 - r * r) / np.sqrt(nw), (i, j, ww[i, j])
    sd = np.sqrt(np.diag(ee))
    for i in range(4):
        n_eff = n * (1 - PHI[i]) / (1 + PHI[i])
        assert abs(mean[i]) < 4 * SIGMA[i] / np.sqrt(n_eff), i
        assert abs(ee[i, i] / SIGMA[i] ** 2 - 1) < 4 * np.sqrt(2 / n_eff), i
        for j in range(i):
            want = CORR[i, j] * np.sqrt((1 - PHI[i] ** 2) * (1 - PHI[j] ** 2)) / (1 - PHI[i] * PHI[j])
            got = ee[i, j] / (sd[i] * sd[j])
            # the sample correlation of two AR(1) series: variance about (1 + phi_i phi_j)/(1 - phi_i phi_j) / n
            # times (1 - rho^2)^2, taken without the last factor
            se = np.sqrt((1 + PHI[i] * PHI[j]) / (1 - PHI[i] * PHI[j]) / n)
            assert abs(got - want) < 4 * se, (i, j, got, want)


def test_bilinear_columns_correlate_by_their_shared_weights(host):
    """cells sharing bilinear nodes correlate by sum w_a w_b over the shared ids; the lognormal mean is kept with mixed
    weights"""
    seed, nrec, phi, nrep = 99, 3000, [0.0, 0.0, 0.8, 0.5], 20
    sigma = [1.0, 1.0, 1.0, 0.4]
    ny = nx = 16
    basis, w = api.bilinear_noise_basis(ny, nx, 4)   # a 5 x 5 lattice of nodes
    ids = np.unique(basis)
    idx = np.searchsorted(ids, basis).astype(np.int32)
    cell = {"a": 1 * nx + 1, "same": 2 * nx + 3, "part": 1 * nx + 6, "none": 1 * nx + 9}
    pairs = [("a", "same"), ("a", "part"), ("a", "none")]
    sums = {}
    for rep in range(nrep):   # independent lattices of streams: nrep * 25 basis streams x 3,000 records
        _, E = host.basis_window(seed, sigma, phi, CORR, ids + rep * 1000, 0, 1, nrec)
        e, _, _ = host.mix(idx, w, E[:, 0])
        for x, y in [("a", "a")] + pairs + [(p, p) for _, p in pairs]:
            sums[x, y] = sums.get((x, y), 0.0) + (e[cell[x]] * e[cell[y]]).sum()
        e, q, _ = host.mix(idx, w, E[:, 3])
        m = host.apply_mixed(2, sigma[3], np.ones(e.size), e.ravel(), np.repeat(q, nrec))
        sums["ln"] = sums.get("ln", 0.0) + m.sum()
        sums["ln2"] = sums.get("ln2", 0.0) + (m * m).sum()
    n = nrep * nrec
    wants = []
    for x, y in pairs:
        ca, cb = cell[x], cell[y]
        want = sum(w[ca, i] * w[cb, j] for i in range(4) for j in range(4) if basis[ca, i] == basis[cb, j])
        rho = sums[x, y] / np.sqrt(sums[x, x] * sums[y, y])
        # kind 0 is white noise: the sample correlation has standard error (1 - rho^2) / sqrt(n)
        assert abs(rho - want) < 4 * (1 - want * want) / np.sqrt(n), (x, y, rho, want)
        wants.append(want)
    assert wants[0] > wants[1] > wants[2] == 0.0   # all four nodes shared, two, none
    # lognormal with mixed weights: E[exp(e - q sigma^2 / 2)] = 1 for every cell
    nln = n * basis.shape[0]
    mean = sums["ln"] / nln
    var = sums["ln2"] / nln - mean * mean
    n_eff = nln * (1 - 0.5) / (1 + 0.5) / 16        # AR(0.5), and about 16 cells share each node
    assert abs(mean - 1) < 4 * np.sqrt(var / n_eff), mean


def test_nothing_correlates_across_seeds(host):
    ids = np.arange(10_000)
    _, E1 = host.basis_window(1, [1.0] * 4, [0.0] * 4, CORR, ids, 0, 1, 300)
    _, E2 = host.basis_window(2, [1.0] * 4, [0.0] * 4, CORR, ids, 0, 1, 300)
    n = E1[:, 0].size
    for k in range(4):
        for j in range(4):
            rho = (E1[:, k] * E2[:, j]).mean() / np.sqrt((E1[:, k] ** 2).mean() * (E2[:, j] ** 2).mean())
            assert abs(rho) < 4 / np.sqrt(n), (k, j)


# ---- the cursor rule per basis stream -------------------------------------------------------------------------------
def test_cursor_rule_per_basis_stream_gives_the_pure_function(host):
    """launch windows of random lengths with backward and forward clock jumps, through the four-kind window rule with
    held state: every window equals the pure function of the record"""
    rng = np.random.default_rng(6)
    seed, ids, nrec = 2025, np.array([0, 3, 77, 4096]), 700
    _, pure = host.basis_window(seed, SIGMA, PHI, CORR, ids, 0, 1, nrec)
    state = np.zeros((len(ids), 4, 2))
    cursor, tc = 0, 1
    restarts = jumps = 0
    for _ in range(400):
        u = rng.random()
        if u < 0.05:
            tc = int(rng.integers(1, tc + 1))
            jumps += 1
        elif u < 0.08:
            tc = min(nrec - 30, tc + int(rng.integers(2, 40)))
        first = max(tc - 1, 1)
        last = min(first + int(rng.integers(0, 24)), nrec)
        restarts += not (cursor >= 1 and first >= cursor - 1)
        new, E = host.basis_window(seed, SIGMA, PHI, CORR, ids, cursor, first, last, state)
        assert np.array_equal(bits(E), bits(pure[:, :, first - 1:last])), (cursor, first, last)
        assert new == (cursor if cursor >= 1 and first >= cursor - 1 and cursor > last else last)
        cursor = new
        assert np.array_equal(bits(state[:, :, 1]), bits(pure[:, :, cursor - 1]))
        if cursor > 1:
            assert np.array_equal(bits(state[:, :, 0]), bits(pure[:, :, cursor - 2]))
        tc = last if last < nrec - 30 else 1
    assert restarts > 5 and jumps > 5


# ---- argument rules -------------------------------------------------------------------------------------------------
def test_argument_rules(host):
    ncol, nmix = 5, 3
    ok = dict(sigma=[1.0, 0.5, 0.0, 0.2], phi=[0.5] * 4, mode=[0, 1, 2, 0], corr=CORR, nmix=nmix, ncol=ncol,
              basis=np.arange(ncol * nmix).reshape(ncol, nmix), weight=np.ones((ncol, nmix)))
    on, single, L = host.check(**ok)
    assert on and not single and np.array_equal(bits(L), bits(cref.cholesky(CORR)))
    dup = ok["basis"].copy()
    dup[2, 2] = dup[2, 0]
    empty_dup = ok["basis"].copy()
    empty_dup[1] = [-1, 4, -1]       # -1 may repeat
    assert not isinstance(host.check(**{**ok, "basis": empty_dup}), str)
    asym = CORR.copy()
    asym[0, 1] += 1e-16 * 8
    diag = CORR.copy()
    diag[2, 2] = 1.0 + 2 ** -52
    bad = {
        "sigma": dict(sigma=[np.nan, 1, 1, 1]), "sigma<0": dict(sigma=[1, -0.5, 1, 1]), "sigma inf": dict(sigma=[1, 1, np.inf, 1]),
        "phi": dict(phi=[0.5, 1.0, 0.5, 0.5]), "phi<0": dict(phi=[-0.1, 0.5, 0.5, 0.5]), "mode": dict(mode=[0, 0, 3, 0]),
        "nmix 0": dict(nmix=0), "nmix 9": dict(nmix=9), "id": dict(basis=np.full((ncol, nmix), -2)),
        "duplicate": dict(basis=dup), "weight nan": dict(weight=np.where(np.eye(ncol, nmix) > 0, np.nan, 1.0)),
        "weight inf": dict(weight=np.full((ncol, nmix), -np.inf)), "corr nan": dict(corr=np.where(CORR == 0.5, np.nan, CORR)),
        "asymmetric": dict(corr=asym), "diagonal": dict(corr=diag),
        "singular": dict(corr=np.ones((4, 4))),
        "indefinite": dict(corr=np.array([[1, .9, .9, 0], [.9, 1, -.9, 0], [.9, -.9, 1, 0], [0, 0, 0, 1.0]])),
    }
    for name, kw in bad.items():
        assert isinstance(host.check(**{**ok, **kw}), str), name
    # the single-stream case, and what is not
    s1 = dict(ok, nmix=1, basis=np.arange(ncol), weight=None, corr=None)
    assert host.check(**s1)[1]
    assert host.check(**{**s1, "corr": np.eye(4)})[1]
    assert host.check(**{**s1, "weight": np.ones(ncol)})[1]
    assert not host.check(**{**s1, "weight": np.full(ncol, 2.0)})[1]
    assert not host.check(**{**s1, "corr": EQUICORR})[1]
    assert not host.check(**dict(s1, nmix=2, basis=np.stack([np.arange(ncol), -np.ones(ncol)], 1)))[1]
    # all sigma 0 switches it off
    assert host.check(**{**ok, "sigma": [0.0] * 4})[0] is False


# ---- the bilinear helper --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ny,nx,spacing", [(64, 32, 8), (7, 5, 3), (1, 1, 1), (10, 13, 1), (33, 17, 16)])
def test_bilinear_basis(ny, nx, spacing):
    basis, w = api.bilinear_noise_basis(ny, nx, spacing)
    assert basis.shape == (ny * nx, 4) and basis.dtype == np.int32 and w.shape == (ny * nx, 4)
    assert np.allclose((w * w).sum(1), 1.0, rtol=0, atol=1e-15)
    assert (w >= 0).all()
    assert all(len(set(r)) == 4 for r in basis.tolist())   # distinct ids within a cell
    nxl = (nx - 1) // spacing + 2
    y, x = np.divmod(np.arange(ny * nx), nx)
    on_node = (y % spacing == 0) & (x % spacing == 0)
    # a cell on a lattice node is that node's stream alone
    assert np.array_equal(basis[on_node, 0], (y[on_node] // spacing) * nxl + x[on_node] // spacing)
    assert (w[on_node, 0] == 1.0).all() and (w[on_node, 1:] == 0.0).all()
    # shards take slices of the global arrays: together they are the grid's, ids and weights alike
    for world in (2, 3):
        parts = [distributed.shard(ny * nx, rank, world) for rank in range(world)]
        assert np.array_equal(np.concatenate([basis[c0:c0 + n] for c0, n in parts]), basis)
        assert np.array_equal(np.concatenate([w[c0:c0 + n] for c0, n in parts]), w)


def test_bilinear_basis_rejects_bad_sizes():
    for args in ((0, 4, 2), (4, 4, 0), (4, -1, 2)):
        with pytest.raises(ValueError):
            api.bilinear_noise_basis(*args)
