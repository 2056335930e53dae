"""Correlated stochastic forcing (samsim_b200_set_stochastic_forcing_correlated) on the GPU: the device's noise against
the host build of noise.cuh, the single-stream case against samsim_b200_set_stochastic_forcing bit for bit, parity with
the oracle fed the perturbed series of the numpy reference, and the same bits whatever the launch lengths, re-binning,
statistics, table path, streaming, checkpoints, clock jumps or sharding of a bilinear grid."""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

from samsim_b200 import api, distributed
from oracle import parity_util as pu

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE))
import correlated_ref as cref  # noqa: E402
import scenarios  # noqa: E402
from test_correlated_forcing_cpu import CORR, CorrHost  # noqa: E402
from test_stochastic_forcing_gpu import (MODE, NCOL, NREC, PHI, SEED, SIGMA, STEPS, _all_state, _engine,  # noqa: E402
                                         _raw_differ, _record_aligned_t2m, _run, _setup)

pytestmark = pytest.mark.gpu

NY, NX, SPACING = 64, 32, 8     # NCOL cells, a 9 x 5 lattice of basis streams
BASIS, WEIGHTS = api.bilinear_noise_basis(NY, NX, SPACING)


@pytest.fixture(scope="module")
def host():
    return CorrHost()


def _corr(st, era, site, scale, offset, basis=BASIS, weights=WEIGHTS, sigma=SIGMA, two_pass=False, corr=CORR):
    eng = _engine(st, len(site), two_pass)
    eng.set_forcing(era, site, scale, offset)
    eng.set_stochastic_forcing(SEED, sigma, PHI, MODE, corr=corr, basis=basis, weights=weights)
    return eng


@pytest.fixture(scope="module")
def corr_run():
    """the reference of the invariance tests: one handle, the bilinear grid, the uneven launches of STEPS"""
    st, era, site, scale, offset = _setup()
    eng = _run(_corr(st, era, site, scale, offset))
    assert (eng.status() == 0).all()
    return _all_state(eng), eng.get_clock()


def _same_as(run, eng):
    state, clock = run
    assert eng.get_clock() == clock
    assert (eng.status() == 0).all()
    bad = _raw_differ(state, _all_state(eng))
    assert not bad, bad


def _mixed_columns(ncol, nmix, pool, seed):
    """basis[ncol, nmix] of distinct ids from `pool` with about a quarter empty, normal (signed) weights"""
    rng = np.random.default_rng(seed)
    basis = np.stack([rng.choice(pool, nmix, replace=False) for _ in range(ncol)]).astype(np.int32)
    basis[rng.random(basis.shape) < 0.25] = -1
    return basis, rng.normal(size=basis.shape)


# ---- 1. the generator on the device --------------------------------------------------------------------------------
def test_device_noise_equals_host_build(host):
    st = scenarios.sheba_state(200)
    ncol, nrec = 4096, 3000
    pool = np.random.default_rng(2).choice(2 ** 31 - 1, 300, replace=False)
    pool[:2] = [0, 2 ** 31 - 1]
    basis, w = _mixed_columns(ncol, 4, pool, 3)
    basis[7] = -1                                  # a column with no entry
    eng = _engine(st, ncol)
    sigma = [0.3, 0.0, 2.0, 0.8]
    eng.set_stochastic_forcing(SEED, sigma, PHI, [1, 0, 0, 2], corr=CORR, basis=basis, weights=w)
    ids = np.unique(basis[basis >= 0])
    _, E = host.basis_window(SEED, sigma, PHI, CORR, ids, 0, 1, nrec)   # [nb, 4, nrec]
    idx = np.where(basis >= 0, np.searchsorted(ids, basis), -1).astype(np.int32)
    for k in range(4):
        want = np.zeros((ncol, nrec)) if sigma[k] == 0.0 else host.mix(idx, w, E[:, k])[0]
        got = eng.forcing_noise(k, 1, nrec)
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), k
        if k == 2:
            assert np.array_equal(eng.forcing_noise(2, 1501, 77, col0=1000, n=33), want[1000:1033, 1500:1577])
            assert (got[7] == 0).all()


# ---- 2. the single-stream case -------------------------------------------------------------------------------------
def test_single_stream_case_gives_the_bits_of_set_stochastic_forcing():
    """nmix 2 with the second entry empty and weights 1.0 runs the two-kernel path; it gives the bits of
    set_stochastic_forcing with the same streams, in state and in forcing_noise"""
    st, era, site, scale, offset = _setup()
    streams = np.arange(NCOL, dtype=np.int32) // 3
    streams[::11] = -1
    a = _engine(st, NCOL)
    a.set_forcing(era, site, scale, offset)
    a.set_stochastic_forcing(SEED, SIGMA, PHI, MODE, streams)
    b = _engine(st, NCOL)
    b.set_forcing(era, site, scale, offset)
    basis = np.stack([streams, np.full(NCOL, -1, np.int32)], axis=1)
    b.set_stochastic_forcing(SEED, SIGMA, PHI, MODE, corr=np.eye(4), basis=basis, weights=np.ones((NCOL, 2)))
    for k in range(4):
        na, nb = a.forcing_noise(k, 1, 300), b.forcing_noise(k, 1, 300)
        assert np.array_equal(na.view(np.int64), nb.view(np.int64)), k
    _run(a)
    _run(b)
    assert a.get_clock() == b.get_clock()
    bad = _raw_differ(_all_state(a), _all_state(b))
    assert not bad, bad


# ---- 3. parity with the oracle ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mixed_oracles(oracle_mod, host):
    """16 oracle columns of the bilinear grid, each fed its perturbed series from the numpy reference"""
    st, era, site, scale, offset = _setup()
    sample = np.sort(np.random.default_rng(9).choice(NCOL, 16, replace=False))
    values = np.stack([era[site[c]] * scale[:, c, None] + offset[:, c, None] for c in sample])   # [16, 4, NREC]
    pert = cref.perturbed(SEED, SIGMA, PHI, MODE, CORR, BASIS[sample], WEIGHTS[sample], values, host.det_log,
                          host.det_cos, host.det_exp)
    cols = []
    for q in range(len(sample)):
        col = oracle_mod.Column(4, "det")
        col.set_forcing(*[pert[q, k] for k in range(4)])
        col.load_state(st)
        cols.append(col)
    assert oracle_mod.run_batch(cols, sum(STEPS), os.cpu_count() or 1) == 0
    return sample, cols


@pytest.mark.parametrize("two_pass", [False, True])
def test_parity_with_the_oracle(mixed_oracles, two_pass):
    sample, cols = mixed_oracles
    st, era, site, scale, offset = _setup()
    eng = _run(_corr(st, era, site, scale, offset, two_pass=two_pass))
    for c, col in zip(sample, cols):
        bad = pu.compare_column(col, eng, int(c), label=f"column {c}: ")
        assert not bad, "\n".join(bad[:12])
        assert col.events() == eng.events(int(c)) - scenarios.DEVICE_ONLY, (c, sorted(col.events() ^ eng.events(int(c))))


# ---- 4. the record value the step reads -----------------------------------------------------------------------------
def test_snapshot_t2m_is_the_perturbed_record(host):
    st, era, site, scale, offset = _setup()
    basis = BASIS.copy()
    basis[::7] = -1
    eng = _corr(st, era, site, scale, offset, basis=basis)
    eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    recs = _record_aligned_t2m(eng, 3)
    last = recs[-1][0]
    values = np.stack([era[site[c]][:, :last] * scale[:, c, None] + offset[:, c, None] for c in range(NCOL)])
    pert = cref.perturbed(SEED, SIGMA, PHI, MODE, CORR, basis, WEIGHTS, values, host.det_log, host.det_cos,
                          host.det_exp)
    for tc, t2m in recs:
        assert np.array_equal(t2m.view(np.int64), pert[:, 2, tc - 1].view(np.int64)), tc
        assert np.array_equal(t2m[::7].view(np.int64), values[::7, 2, tc - 1].view(np.int64))


def test_empty_columns_and_sigma_zero_kinds_read_the_plain_record():
    st, era, site, scale, offset = _setup()
    a = _engine(st, NCOL)
    a.set_forcing(era, site, scale, offset)
    basis = BASIS.copy()
    basis[: NCOL // 4] = -1
    b = _corr(st, era, site, scale, offset, basis=basis, sigma=[0.3, 10.0, 0.0, 0.5])
    for eng in (a, b):
        eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    ra, rb = _record_aligned_t2m(a, 2), _record_aligned_t2m(b, 2)
    for (ta, xa), (tb, xb) in zip(ra, rb):
        assert ta == tb and np.array_equal(xa.view(np.int64), xb.view(np.int64))
    assert (b.forcing_noise(2, 1, 100) == 0).all() and (b.forcing_noise(1, 1, 100)[: NCOL // 4] == 0).all()
    # all-empty columns match a run without the feature in every raw bit
    _run(a, STEPS[:3])
    _run(b, STEPS[:3])
    ctl = NCOL // 4
    bad = _raw_differ(_all_state(a, 0, ctl), _all_state(b, 0, ctl))
    assert not bad, bad
    assert not pu.same_bits(a.get_scalar("fl_lw")[ctl:], b.get_scalar("fl_lw")[ctl:]).all()


# ---- 5. the same bits as one plain run -----------------------------------------------------------------------------
def test_launch_lengths(corr_run):
    st, era, site, scale, offset = _setup()
    _same_as(corr_run, _run(_corr(st, era, site, scale, offset), (sum(STEPS),)))
    _same_as(corr_run, _run(_corr(st, era, site, scale, offset), (1, 1, 1, 1079, 1080, 2, 6577)))


def test_rebinning(corr_run):
    st, era, site, scale, offset = _setup()
    a = _corr(st, era, site, scale, offset)
    a.step(700)
    assert a.rebin()
    _run(a, (3334, 4610, 97))
    _same_as(corr_run, a)
    b = _corr(st, era, site, scale, offset)
    b.set_rebin_interval(1500)
    _run(b)
    assert b.divergence()["rebins"] >= 1
    _same_as(corr_run, b)


def test_group_and_time_statistics_on(corr_run):
    st, era, site, scale, offset = _setup()
    eng = _corr(st, era, site, scale, offset)
    eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    eng.set_group_stats(site, max_records=8)
    eng.set_time_stats(1, None, max_windows=8)
    _run(eng)
    assert eng.group_stats_held() == 2 and eng.time_stats_held() == 2
    _same_as(corr_run, eng)


def test_global_table_equals_staged_table(corr_run):
    st, era, site, scale, offset = _setup()
    perm = np.random.default_rng(4).permutation(NCOL).astype(np.int32)
    table = np.empty((NCOL, 4, NREC))
    table[perm] = era[site]
    eng = _engine(st, NCOL)
    eng.set_forcing(table, perm, scale, offset)
    eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE, corr=CORR, basis=BASIS, weights=WEIGHTS)
    _same_as(corr_run, _run(eng))


def test_update_forcing_records_mid_run(corr_run):
    st, era, site, scale, offset = _setup()
    partial = era.copy()
    partial[:, :, 1597:] = np.nan
    eng = _corr(st, partial, site, scale, offset)
    eng.step(701)
    eng.update_forcing_records(1598, era[:, :, 1597:1620])
    _run(eng, (3333, 4610, 97))
    _same_as(corr_run, eng)


def test_checkpoint_mid_run(corr_run, tmp_path):
    st, era, site, scale, offset = _setup()
    a = _corr(st, era, site, scale, offset)
    _run(a, (1, 700, 3333))
    ck = tmp_path / "mid.ck"
    a.save_checkpoint(ck)
    b = _corr(st, era, site, scale, offset)
    b.load_checkpoint(ck)
    _same_as(corr_run, _run(b, (4610, 97)))
    a.step(5000)
    a.load_checkpoint(ck)
    _same_as(corr_run, _run(a, (4610, 97)))


def test_clock_back_and_forward(corr_run, tmp_path):
    st, era, site, scale, offset = _setup()
    eng = _corr(st, era, site, scale, offset)
    _run(eng, (1, 700))
    ck = tmp_path / "c.ck"
    eng.save_checkpoint(ck)
    clk = eng.get_clock()
    eng.set_clock(clk["time"] + 30 * 10800.0, clk["i"], clk["n_time_out"], clk["time_counter"] + 30)
    eng.step(3)
    eng.load_checkpoint(ck)
    eng.set_clock(clk["time"] - 40 * 10800.0, clk["i"], clk["n_time_out"], clk["time_counter"] - 40)
    eng.set_clock(clk["time"], clk["i"], clk["n_time_out"], clk["time_counter"])
    _same_as(corr_run, _run(eng, (3333, 4610, 97)))


def test_two_shards_split_the_bilinear_grid(corr_run):
    """the shard boundary is cell row 32, a lattice row: the nodes of row 4 feed cells on both shards"""
    st, era, site, scale, offset = _setup()
    state, clock = corr_run
    shared = None
    for rank in range(2):
        col0, n = distributed.shard(NCOL, rank, 2)
        ids = set(BASIS[col0:col0 + n][WEIGHTS[col0:col0 + n] > 0].tolist())
        shared = ids if shared is None else shared & ids
        eng = _engine(st, n)
        eng.set_forcing(era, site[col0:col0 + n], scale[:, col0:col0 + n], offset[:, col0:col0 + n])
        eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE, corr=CORR, basis=BASIS[col0:col0 + n],
                                   weights=WEIGHTS[col0:col0 + n])
        _run(eng)
        assert eng.get_clock() == clock
        mine = {k: v[col0:col0 + n] for k, v in state.items()}
        bad = _raw_differ(mine, _all_state(eng))
        assert not bad, (rank, bad)
    assert len(shared) >= 5


def test_one_setting_one_state():
    """each setter replaces the other's setting"""
    st, era, site, scale, offset = _setup(256)
    eng = _engine(st, 256)
    eng.set_forcing(era, site, scale, offset)
    eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE)
    plain = eng.forcing_noise(1, 1, 30)
    eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE, corr=CORR, basis=BASIS[:256], weights=WEIGHTS[:256])
    mixed = eng.forcing_noise(1, 1, 30)
    assert not np.array_equal(plain, mixed)
    eng.step(1100)
    eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE)
    assert np.array_equal(eng.forcing_noise(1, 1, 30), plain)
    eng.step(1100)
    assert (eng.status() == 0).all()


# ---- 6. arguments and config -----------------------------------------------------------------------------------------
def test_arguments_and_config():
    st, era, site, scale, offset = _setup(256)
    eng = _corr(st, era, site, scale, offset, basis=BASIS[:256], weights=WEIGHTS[:256])
    before = [eng.forcing_noise(k, 1, 40) for k in range(4)]
    L, h = eng.L, eng.h
    ok = dict(sigma=np.array([2.0, 1.0, 1.0, 1.0]), phi=np.full(4, 0.5), mode=np.zeros(4, np.int32), corr=CORR.copy(),
              nmix=4, basis=BASIS[:256].copy(), weights=WEIGHTS[:256].copy())
    dup = ok["basis"].copy()
    dup[5, 3] = dup[5, 1]
    asym = CORR.copy()
    asym[1, 0] = np.nextafter(asym[1, 0], 1.0)
    diag = CORR.copy()
    diag[3, 3] = 0.999
    bad = [
        dict(sigma=np.array([np.nan, 1, 1, 1.0])), dict(sigma=np.array([1, -0.5, 1, 1.0])),
        dict(phi=np.array([0.5, 1.0, 0.5, 0.5])), dict(mode=np.array([0, 0, 3, 0], np.int32)),
        dict(nmix=0), dict(nmix=9, basis=np.full((256, 9), -1, np.int32), weights=np.ones((256, 9))),
        dict(basis=np.full((256, 4), -2, np.int32)), dict(basis=dup),
        dict(weights=np.where(np.arange(1024).reshape(256, 4) == 77, np.inf, 1.0)),
        dict(corr=np.where(CORR == 0.5, np.nan, CORR)), dict(corr=asym), dict(corr=diag), dict(corr=np.ones((4, 4))),
        dict(basis=None),
    ]
    for kw in bad:
        a = ok | kw
        b = None if a["basis"] is None else np.ascontiguousarray(a["basis"], np.int32)
        w = np.ascontiguousarray(a["weights"], np.float64)
        cr = np.ascontiguousarray(a["corr"], np.float64)
        rc = L.samsim_b200_set_stochastic_forcing_correlated(h, 1, api._dp(a["sigma"]), api._dp(a["phi"]),
                                                             api._ip(a["mode"]), api._dp(cr), a["nmix"], api._ip(b),
                                                             api._dp(w))
        assert rc == -1, list(kw)
        for k in range(4):   # the previous setting is kept
            assert np.array_equal(eng.forcing_noise(k, 1, 40), before[k]), list(kw)
    with pytest.raises(ValueError):
        eng.set_stochastic_forcing(1, ok["sigma"], ok["phi"], ok["mode"], np.arange(256), basis=ok["basis"])
    eng.step(50)
    # all sigma 0 switches it off
    eng.set_stochastic_forcing(1, [0.0] * 4, [0.5] * 4, [0] * 4, corr=CORR, basis=BASIS[:256])
    assert (eng.forcing_noise(1, 1, 40) == 0).all()
    eng.step(50)
    assert (eng.status() == 0).all()
    lab = api.Engine(api.Config.from_state({**st, "atmoflux_flag": 1}), 8)
    with pytest.raises(api.SamsimError) as e:
        lab.set_stochastic_forcing(1, [1.0] * 4, [0.5] * 4, [0] * 4, corr=CORR)
    assert e.value.code == -4


# ---- 7. a large batch -----------------------------------------------------------------------------------------------
def test_million_columns_with_4096_basis_streams():
    """1,048,576 columns mixing 4 of 4,096 basis streams step through a record; the snapshot T2m at the record equals
    the plain record plus get_forcing_noise on sampled columns"""
    st = scenarios.sheba_state(200)
    era = np.load(scenarios.GOLDEN / "forcing_era.npz")
    series = np.asarray(era[str(era["sites"][0])][:, :NREC])[None]   # one site
    ncol = 1 << 20
    c = np.arange(ncol)
    basis = np.stack([(c + m * 1024) % 4096 for m in range(4)], axis=1).astype(np.int32)
    w = np.random.default_rng(7).normal(size=basis.shape)
    eng = _engine(st, ncol)
    eng.set_forcing(series)
    eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE, corr=CORR, basis=basis, weights=w)
    eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    (tc, t2m), = _record_aligned_t2m(eng, 1)
    assert (eng.status() == 0).all()
    for col0 in (0, 4095, 524_288, ncol - 100):
        e = eng.forcing_noise(2, tc, 1, col0=col0, n=100)[:, 0]
        want = series[0, 2, tc - 1] + e
        assert np.array_equal(t2m[col0:col0 + 100].view(np.int64), want.view(np.int64)), col0
        assert np.std(e) > 0.3 * SIGMA[2]   # perturbed: four unit-variance streams with normal weights
