"""Stochastic forcing perturbations (samsim_b200_set_stochastic_forcing) on the GPU: the device's noise against the host
build of noise.cuh, parity with the oracle fed the perturbed series of the numpy reference, and the same bits whatever
the launch lengths, re-binning, statistics, table path, streaming, checkpoints, clock jumps or sharding."""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

from samsim_b200 import api, distributed
from oracle import parity_util as pu

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE))
import scenarios  # noqa: E402
import stochastic_ref as ref  # noqa: E402
from test_stochastic_forcing_cpu import Host, build_lib  # noqa: E402

pytestmark = pytest.mark.gpu

NREC = 2928
NCOL = 2048
SEED = 0x5EED_0F_F0_4C1
# additive SW would be unphysical at night: multiplicative SW, additive LW and T2m, lognormal precip
SIGMA = [0.25, 12.0, 1.5, 0.6]
PHI = [0.7, 0.8, 0.9, 0.5]
MODE = [1, 0, 0, 2]
STEPS = (1, 700, 3333, 4610, 97)   # uneven launches across record boundaries and two output steps


@pytest.fixture(scope="module")
def host():
    return Host(build_lib())


def _era_sites() -> np.ndarray:
    z = np.load(scenarios.GOLDEN / "forcing_era.npz")
    return np.stack([z[str(s)][:, :NREC] for s in z["sites"]])   # [9, 4, NREC]


def _perturbations(ncol, seed):
    rng = np.random.default_rng(seed)
    scale = np.ones((4, ncol))
    offset = np.zeros((4, ncol))
    scale[0], scale[1], scale[3] = rng.uniform(0.9, 1.1, ncol), rng.uniform(0.95, 1.05, ncol), rng.uniform(0.5, 1.5, ncol)
    offset[2] = rng.uniform(-2, 2, ncol)
    return scale, offset


def _setup(ncol=NCOL):
    st = scenarios.sheba_state(200)
    site = (np.arange(ncol) % 9).astype(np.int32)
    scale, offset = _perturbations(ncol, 3)
    return st, _era_sites(), site, scale, offset


def _engine(st, ncol, two_pass=False):
    eng = api.Engine(api.Config.from_state(st), ncol)
    eng.load_column_state(st, 0)
    eng.broadcast_column(0, 0, ncol)
    eng.set_tuning(two_pass)
    eng.clear_events()
    return eng


def _plain(st, era, site, scale, offset, streams=None, sigma=SIGMA, two_pass=False):
    eng = _engine(st, len(site), two_pass)
    eng.set_forcing(era, site, scale, offset)
    if streams is not False:
        eng.set_stochastic_forcing(SEED, sigma, PHI, MODE, streams)
    return eng


def _all_state(eng, col0=0, n=None):
    d = {nm: eng.get_array(nm, col0, n) for nm in pu.CMP_ARRAYS}
    d.update({nm: eng.get_scalar(nm, col0, n) for nm in api.SCALAR_IDS})
    d.update({nm: eng.get_int(nm, col0, n) for nm in api.INT_IDS})
    return d


def _raw_differ(a, b):
    """names whose raw bits differ (+0.0 and -0.0 differ here)"""
    return [n for n in a if not np.array_equal(np.ascontiguousarray(a[n]).view(np.uint8), np.ascontiguousarray(b[n]).view(np.uint8))]


def _run(eng, steps=STEPS):
    for n in steps:
        eng.step(n)
    return eng


@pytest.fixture(scope="module")
def plain_run():
    """the reference of the invariance tests: one handle, the uneven launches of STEPS"""
    st, era, site, scale, offset = _setup()
    eng = _run(_plain(st, era, site, scale, offset))
    assert (eng.status() == 0).all()
    return _all_state(eng), eng.get_clock()


def _same_as_plain(plain_run, eng):
    state, clock = plain_run
    assert eng.get_clock() == clock
    assert (eng.status() == 0).all()
    bad = _raw_differ(state, _all_state(eng))
    assert not bad, bad


# ---- 1. the generator on the device --------------------------------------------------------------------------------
def test_device_noise_equals_host_build(host):
    st = scenarios.sheba_state(200)
    ncol = 4096
    rng = np.random.default_rng(1)
    streams = rng.integers(0, 1 << 31, ncol).astype(np.int32)
    streams[:5] = [0, 1, 2, 2 ** 31 - 1, -1]
    streams[100:200] = streams[50]                       # shared streams
    eng = _engine(st, ncol)
    sigma = [0.3, 0.0, 2.0, 0.8]
    want = []
    for k in range(4):
        w = host.series(SEED, sigma[k], PHI[k], k, np.maximum(streams, 0), 1, 3000)
        w[streams < 0] = 0.0
        want.append(np.zeros_like(w) if sigma[k] == 0.0 else w)
    for mode in ([0, 0, 0, 0], [1, 2, 0, 2], [2, 1, 1, 1]):   # the mode changes what the step reads, not e
        eng.set_stochastic_forcing(SEED, sigma, PHI, mode, streams)
        for k in range(4):
            got = eng.forcing_noise(k, 1, 3000)
            assert np.array_equal(got.view(np.int64), want[k].view(np.int64)), (mode, k)
    # a sub-range of records and columns is the same function
    got = eng.forcing_noise(2, 1501, 77, col0=1000, n=33)
    assert np.array_equal(got, host.series(SEED, sigma[2], PHI[2], 2, streams[1000:1033], 1501, 77))
    # NULL streams: the caller column
    eng.set_stochastic_forcing(SEED, sigma, PHI, [0] * 4)
    assert np.array_equal(eng.forcing_noise(3, 1, 50), host.series(SEED, sigma[3], PHI[3], 3, np.arange(ncol), 1, 50))


# ---- 2. parity with the oracle ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def noisy_oracles(oracle_mod, host):
    """16 oracle columns, each fed its perturbed series from the numpy reference, advanced two model days"""
    st, era, site, scale, offset = _setup()
    sample = np.sort(np.random.default_rng(8).choice(NCOL, 16, replace=False))
    values = np.stack([era[site[c]] * scale[:, c, None] + offset[:, c, None] for c in sample])   # [16, 4, NREC]
    pert = ref.perturbed(SEED, SIGMA, PHI, MODE, sample, values, host.det_log, host.det_cos, host.det_exp)
    cols = []
    for q in range(len(sample)):
        col = oracle_mod.Column(4, "det")
        col.set_forcing(*[pert[q, k] for k in range(4)])
        col.load_state(st)
        cols.append(col)
    assert oracle_mod.run_batch(cols, sum(STEPS), os.cpu_count() or 1) == 0
    return sample, cols


@pytest.mark.parametrize("two_pass", [False, True])
def test_parity_with_the_oracle(noisy_oracles, two_pass):
    sample, cols = noisy_oracles
    st, era, site, scale, offset = _setup()
    eng = _run(_plain(st, era, site, scale, offset, two_pass=two_pass))
    for c, col in zip(sample, cols):
        bad = pu.compare_column(col, eng, int(c), label=f"column {c}: ")
        assert not bad, "\n".join(bad[:12])
        assert col.events() == eng.events(int(c)) - scenarios.DEVICE_ONLY, (c, sorted(col.events() ^ eng.events(int(c))))


# ---- 3. the record value the step reads -----------------------------------------------------------------------------
def _record_aligned_t2m(eng, nrec_ahead):
    """step to the start of the next nrec_ahead records; at each, make the step an output step and read the snapshot's
    T2m (the step with time == time_input(tc) takes record tc without interpolation)"""
    out = []
    for _ in range(nrec_ahead):
        clk = eng.get_clock()
        tc = clk["time_counter"] + (1 if clk["time"] > (clk["time_counter"] - 1) * 10800.0 else 0)
        n = int(round(((tc - 1) * 10800.0 - clk["time"]) / 10.0))
        if n > 0:
            eng.step(n)
        clk = eng.get_clock()
        assert clk["time"] == (tc - 1) * 10800.0
        eng.set_clock(clk["time"], clk["i"], eng.cfg.i_time_out, clk["time_counter"])
        eng.step(1)
        out.append((tc, eng.get_snapshot(arrays=False)["T2m"].copy()))
    return out


def test_snapshot_t2m_is_the_perturbed_record(host):
    st, era, site, scale, offset = _setup()
    streams = np.arange(NCOL, dtype=np.int32)
    streams[::7] = -1
    eng = _plain(st, era, site, scale, offset, streams)
    eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    recs = _record_aligned_t2m(eng, 3)
    last = recs[-1][0]
    values = np.stack([era[site[c]][:, :last] * scale[:, c, None] + offset[:, c, None] for c in range(NCOL)])
    pert = ref.perturbed(SEED, SIGMA, PHI, MODE, streams, values, host.det_log, host.det_cos, host.det_exp)
    for tc, t2m in recs:
        assert np.array_equal(t2m.view(np.int64), pert[:, 2, tc - 1].view(np.int64)), tc
        assert np.array_equal(t2m[::7].view(np.int64), values[::7, 2, tc - 1].view(np.int64))


def test_sigma_zero_kind_reads_the_plain_record():
    st, era, site, scale, offset = _setup()
    a = _plain(st, era, site, scale, offset, streams=False)
    b = _plain(st, era, site, scale, offset, sigma=[0.3, 10.0, 0.0, 0.5])
    for eng in (a, b):
        eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    ra, rb = _record_aligned_t2m(a, 2), _record_aligned_t2m(b, 2)
    for (ta, xa), (tb, xb) in zip(ra, rb):
        assert ta == tb and np.array_equal(xa.view(np.int64), xb.view(np.int64))
    assert not np.array_equal(a.get_scalar("fl_lw"), b.get_scalar("fl_lw"))
    assert (b.forcing_noise(2, 1, 100) == 0).all()


# ---- 4. the same bits as one plain run -----------------------------------------------------------------------------
def test_launch_lengths(plain_run):
    st, era, site, scale, offset = _setup()
    _same_as_plain(plain_run, _run(_plain(st, era, site, scale, offset), (sum(STEPS),)))
    _same_as_plain(plain_run, _run(_plain(st, era, site, scale, offset), (1, 1, 1, 1079, 1080, 2, 6577)))


def test_rebinning(plain_run):
    st, era, site, scale, offset = _setup()
    a = _plain(st, era, site, scale, offset)
    a.step(700)
    assert a.rebin()
    _run(a, (3334, 4610, 97))
    _same_as_plain(plain_run, a)
    b = _plain(st, era, site, scale, offset)
    b.set_rebin_interval(1500)
    _run(b)
    assert b.divergence()["rebins"] >= 1
    _same_as_plain(plain_run, b)


def test_group_and_time_statistics_on(plain_run):
    st, era, site, scale, offset = _setup()
    eng = _plain(st, era, site, scale, offset)
    eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    eng.set_group_stats(site, max_records=8)
    eng.set_time_stats(1, None, max_windows=8)
    _run(eng)
    assert eng.group_stats_held() == 2 and eng.time_stats_held() == 2
    _same_as_plain(plain_run, eng)


def test_global_table_equals_staged_table(plain_run):
    st, era, site, scale, offset = _setup()
    perm = np.random.default_rng(4).permutation(NCOL).astype(np.int32)
    table = np.empty((NCOL, 4, NREC))
    table[perm] = era[site]
    eng = _engine(st, NCOL)
    eng.set_forcing(table, perm, scale, offset)
    eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE)
    _same_as_plain(plain_run, _run(eng))


def test_update_forcing_records_mid_run(plain_run):
    st, era, site, scale, offset = _setup()
    partial = era.copy()
    partial[:, :, 1597:] = np.nan
    eng = _engine(st, NCOL)
    eng.set_forcing(partial, site, scale, offset)
    eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE)
    eng.step(701)
    eng.update_forcing_records(1598, era[:, :, 1597:1620])
    _run(eng, (3333, 4610, 97))
    _same_as_plain(plain_run, eng)


def test_checkpoint_mid_run(plain_run, tmp_path):
    st, era, site, scale, offset = _setup()
    a = _plain(st, era, site, scale, offset)
    _run(a, (1, 700, 3333))
    ck = tmp_path / "mid.ck"
    a.save_checkpoint(ck)
    b = _plain(st, era, site, scale, offset)
    b.load_checkpoint(ck)
    _same_as_plain(plain_run, _run(b, (4610, 97)))
    # the same handle after it ran on: the clock moves back, the window restarts from record 1
    a.step(5000)
    a.load_checkpoint(ck)
    _same_as_plain(plain_run, _run(a, (4610, 97)))


def test_clock_back_and_forward(plain_run, tmp_path):
    st, era, site, scale, offset = _setup()
    eng = _plain(st, era, site, scale, offset)
    _run(eng, (1, 700))
    ck = tmp_path / "c.ck"
    eng.save_checkpoint(ck)
    clk = eng.get_clock()
    # forward 30 records (the window resumes and skips records), a few steps, then back through the checkpoint
    eng.set_clock(clk["time"] + 30 * 10800.0, clk["i"], clk["n_time_out"], clk["time_counter"] + 30)
    eng.step(3)
    eng.load_checkpoint(ck)
    # back 40 records and forward again before the next launch: nothing ran in between
    eng.set_clock(clk["time"] - 40 * 10800.0, clk["i"], clk["n_time_out"], clk["time_counter"] - 40)
    eng.set_clock(clk["time"], clk["i"], clk["n_time_out"], clk["time_counter"])
    _same_as_plain(plain_run, _run(eng, (3333, 4610, 97)))


def test_two_shards_with_global_streams(plain_run):
    st, era, site, scale, offset = _setup()
    state, clock = plain_run
    for rank in range(2):
        col0, n = distributed.shard(NCOL, rank, 2)
        eng = _engine(st, n)
        eng.set_forcing(era, site[col0:col0 + n], scale[:, col0:col0 + n], offset[:, col0:col0 + n])
        eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE, distributed.noise_streams(NCOL, rank, 2))
        _run(eng)
        assert eng.get_clock() == clock
        mine = {k: v[col0:col0 + n] for k, v in state.items()}
        bad = _raw_differ(mine, _all_state(eng))
        assert not bad, (rank, bad)


# ---- 5. unperturbed and shared streams --------------------------------------------------------------------------------
def test_stream_minus_one_equals_no_feature_and_shared_streams_agree():
    st, era, site, scale, offset = _setup()
    # columns 2j and 2j+1 read the same site, scale and offset
    site2 = site[np.arange(NCOL) // 2]
    scale2, offset2 = scale[:, np.arange(NCOL) // 2], offset[:, np.arange(NCOL) // 2]
    streams = (np.arange(NCOL) // 2).astype(np.int32)
    streams[: NCOL // 4] = -1
    a = _run(_plain(st, era, site2, scale2, offset2, streams=False))
    b = _run(_plain(st, era, site2, scale2, offset2, streams=streams))
    ctl = NCOL // 4
    bad = _raw_differ(_all_state(a, 0, ctl), _all_state(b, 0, ctl))
    assert not bad, bad
    sb = _all_state(b)
    bad = [k for k, v in sb.items() if _raw_differ({k: v[ctl::2]}, {k: v[ctl + 1::2]})]
    assert not bad, bad
    sa = _all_state(a)
    assert not pu.same_bits(sa["T"][ctl:], sb["T"][ctl:]).all()   # the perturbed ones moved


# ---- 6. arguments and config -----------------------------------------------------------------------------------------
def test_arguments_and_config():
    st, era, site, scale, offset = _setup(256)
    eng = _plain(st, era, site, scale, offset)
    before = [eng.forcing_noise(k, 1, 40) for k in range(4)]
    bad = [
        (dict(sigma=[np.nan, 1, 1, 1]), -1), (dict(sigma=[1, -0.5, 1, 1]), -1), (dict(sigma=[1, 1, np.inf, 1]), -1),
        (dict(phi=[0.5, 1.0, 0.5, 0.5]), -1), (dict(phi=[-0.1, 0.5, 0.5, 0.5]), -1), (dict(phi=[np.nan] * 4), -1),
        (dict(mode=[0, 0, 3, 0]), -1), (dict(mode=[-1, 0, 0, 0]), -1),
        (dict(streams=np.full(256, -2, dtype=np.int32)), -1),
    ]
    for kw, code in bad:
        args = dict(sigma=[2.0, 1.0, 1.0, 1.0], phi=[0.5] * 4, mode=[0] * 4, streams=None) | kw
        with pytest.raises(api.SamsimError) as e:
            eng.set_stochastic_forcing(1, args["sigma"], args["phi"], args["mode"], args["streams"])
        assert e.value.code == code, kw
        for k in range(4):   # the previous setting is kept
            assert np.array_equal(eng.forcing_noise(k, 1, 40), before[k]), kw
    L, h = eng.L, eng.h
    z = np.zeros(4)
    assert L.samsim_b200_set_stochastic_forcing(h, 1, None, api._dp(z), api._ip(np.zeros(4, np.int32)), None) == -1
    out = np.empty(10)
    assert L.samsim_b200_get_forcing_noise(h, 4, 1, 10, 0, 1, api._dp(out)) == -1
    assert L.samsim_b200_get_forcing_noise(h, 0, 0, 10, 0, 1, api._dp(out)) == -1
    assert L.samsim_b200_get_forcing_noise(h, 0, 1, 10, 250, 7, api._dp(out)) == -1
    assert L.samsim_b200_get_forcing_noise(h, 0, 1, 10, 0, 1, None) == -1
    eng.step(50)
    # all sigma 0 switches it off: the step reads the table, the noise reads 0
    eng.set_stochastic_forcing(1, [0.0] * 4, [0.5] * 4, [0] * 4)
    assert (eng.forcing_noise(1, 1, 40) == 0).all()
    eng.step(50)
    assert (eng.status() == 0).all()
    # without atmoflux_flag 2
    lab = api.Engine(api.Config.from_state({**st, "atmoflux_flag": 1}), 8)
    with pytest.raises(api.SamsimError) as e:
        lab.set_stochastic_forcing(1, [1.0] * 4, [0.5] * 4, [0] * 4)
    assert e.value.code == -4
