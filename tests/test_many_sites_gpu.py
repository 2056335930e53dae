"""Forcing tables of any number of sites (samsim_b200_set_forcing with nsite > 16, read in place from global memory),
the 64-bit re-binning key and samsim_b200_update_forcing_records, on the GPU against the staged path, the oracle and
un-binned handles."""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

from samsim_b200 import api
from oracle import parity_util as pu

sys.path.insert(0, str(Path(__file__).resolve().parent))
import scenarios  # noqa: E402

pytestmark = pytest.mark.gpu

NREC = 2928     # one year of 3-hourly records, the length of every ERA site
NCOL = 4096


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


def _shifted_sites(nsite, seed, max_shift=240):
    """nsite distinct series: ERA site p % 9 started max_shift records earlier or later (a different start date) and
    scaled by its own factors"""
    era = _era_sites()
    rng = np.random.default_rng(seed)
    shift = rng.integers(-max_shift, max_shift + 1, nsite)
    fac = np.stack([rng.uniform(0.9, 1.1, nsite), rng.uniform(0.97, 1.03, nsite), np.ones(nsite), rng.uniform(0.5, 1.5, nsite)], 1)
    return np.stack([np.roll(era[p % 9], shift[p], axis=1) * fac[p][:, None] for p in range(nsite)])


def _engine(st, ncol, two_pass=False, rec_shift=0):
    """ncol columns in state st; rec_shift: the clock moved back by that many records, for a table whose first
    rec_shift records are cut off (the times are exact integers, so this changes no result)"""
    cfg = api.Config.from_state(st)
    eng = api.Engine(cfg, ncol)
    eng.load_column_state(st, 0)
    eng.broadcast_column(0, 0, ncol)
    eng.set_clock(st["time"] - rec_shift * 10800.0, st["i"], st["n_time_out"], st["time_counter"] - rec_shift)
    eng.set_tuning(two_pass)
    return eng


def _all_state(eng):
    d = {n: eng.get_array(n) for n in pu.CMP_ARRAYS}
    d.update({n: eng.get_scalar(n) for n in api.SCALAR_IDS})
    d.update({n: eng.get_int(n) for n in api.INT_IDS})
    return d


def _differ(a, b):
    return [n for n in a if not pu.same_bits(a[n], b[n]).all()]


@pytest.mark.parametrize("two_pass", [False, True])
@pytest.mark.parametrize("rec", [60, 200])
def test_global_table_equals_staged_table(two_pass, rec):
    st = scenarios.sheba_state(rec)
    era = _era_sites()
    site9 = (np.arange(NCOL) % 9).astype(np.int32)
    scale, offset = _perturbations(NCOL, rec)
    perm = np.random.default_rng(rec + 1).permutation(NCOL).astype(np.int32)   # column c reads site perm[c]
    table = np.empty((NCOL, 4, NREC))
    table[perm] = era[site9]
    a, b = _engine(st, NCOL, two_pass), _engine(st, NCOL, two_pass)
    a.set_forcing(era, site9, scale, offset)
    b.set_forcing(table, perm, scale, offset)
    for eng in (a, b):
        eng.set_snapshot_mode(api.SNAP_FULL)
        eng.clear_events()
    # uneven launches across record boundaries (1,080 steps each) and two output steps (the first step, then 8,641)
    for n in (1, 700, 3333, 4610, 97):
        a.step(n)
        b.step(n)
    assert a.get_clock() == b.get_clock()
    assert a.get_clock()["n_time_out"] == 8741 - 8642   # output records at the 1st and the 8,642nd step
    bad = _differ(_all_state(a), _all_state(b))
    assert not bad, bad
    sa, sb = a.get_snapshot(), b.get_snapshot()
    assert not [n for n in sa if not pu.same_bits(sa[n], sb[n]).all()]
    assert (a.status() == 0).all() and a.launch_count() == b.launch_count()


@pytest.fixture(scope="module")
def shifted_oracles(oracle_mod):
    """16 oracle columns, each fed exactly its own series*scale + offset, advanced two model days"""
    st = scenarios.sheba_state(200)
    table = _shifted_sites(NCOL, 5)
    soc = np.random.default_rng(6).permutation(NCOL).astype(np.int32)
    scale, offset = _perturbations(NCOL, 7)
    sample = np.sort(np.random.default_rng(8).choice(NCOL, 16, replace=False))
    cols = []
    for c in sample:
        col = oracle_mod.Column(4, "det")
        col.set_forcing(*[table[soc[c], k] * scale[k, c] + offset[k, c] for k in range(4)])
        col.load_state(st)
        cols.append(col)
    assert oracle_mod.run_batch(cols, 17280, os.cpu_count() or 1) == 0
    return st, table, soc, scale, offset, sample, cols


@pytest.mark.parametrize("two_pass", [False, True])
def test_distinct_sites_match_the_oracle(shifted_oracles, two_pass):
    st, table, soc, scale, offset, sample, cols = shifted_oracles
    eng = _engine(st, NCOL, two_pass)
    eng.set_forcing(table, soc, scale, offset)
    eng.clear_events()
    for n in (5000, 8640, 3640):
        eng.step(n)
    for c, col in zip(sample, cols):
        bad = pu.compare_column(col, eng, int(c), label=f"column {c} (site {soc[c]}): ")
        assert not bad, "\n".join(bad[:12])
        assert col.events() == eng.events(int(c)) - scenarios.DEVICE_ONLY, (c, sorted(col.events() ^ eng.events(int(c))))


def test_rebinning_with_more_than_32_sites():
    st = scenarios.sheba_state(200)
    nsite, ncol = 40, 2048
    table = _shifted_sites(nsite, 9)
    soc = (np.arange(ncol) % nsite).astype(np.int32)
    scale, offset = _perturbations(ncol, 10)
    a, b = _engine(st, ncol), _engine(st, ncol)
    for eng in (a, b):
        eng.set_forcing(table, soc, scale, offset)
    # one state everywhere: the site decides the order, and sites 0 and 32 are different sites
    assert a.rebin()
    col_of_slot = np.argsort(a.slot_map())
    assert (np.diff(soc[col_of_slot]) >= 0).all()
    for eng in (a, b):
        eng.step(3000)
    a.rebin()   # drifted: re-bin again mid-run
    for eng in (a, b):
        eng.step(2000)
    assert b.divergence()["rebins"] == 0
    bad = _differ(_all_state(a), _all_state(b))
    assert not bad, bad


@pytest.mark.parametrize("nsite", [9, 64])
def test_update_forcing_records_streams_a_table(nsite):
    st = scenarios.sheba_state(200)   # time_counter 1594: records 1593 and 1594 are read first
    ncol = 1024
    full = _shifted_sites(nsite, 11)
    soc = (np.arange(ncol) % nsite).astype(np.int32)
    scale, offset = _perturbations(ncol, 12)
    partial = full.copy()
    partial[:, :, 1597:] = np.nan   # records 1598 .. : not there yet
    a, b = _engine(st, ncol), _engine(st, ncol)
    a.set_forcing(full, soc, scale, offset)
    b.set_forcing(partial, soc, scale, offset)
    for rec0, n, steps in ((1598, 3, 1000), (1601, 5, 3000), (1606, 20, 5000)):
        a.step(steps)
        b.step(steps)
        assert b.get_clock()["time_counter"] < rec0   # the new records have not been read yet
        b.update_forcing_records(rec0, full[:, :, rec0 - 1:rec0 - 1 + n])
    a.step(4000)
    b.step(4000)
    assert (b.status() == 0).all()
    bad = _differ(_all_state(a), _all_state(b))
    assert not bad, bad


def test_update_forcing_records_arguments():
    st = scenarios.sheba_state(200)
    eng = _engine(st, 64)
    L, h = eng.L, eng.h
    buf = np.zeros((20, 4, 8))
    assert L.samsim_b200_update_forcing_records(h, 1, 8, api._dp(buf)) == -5   # before set_forcing
    eng.set_forcing(_shifted_sites(20, 13), (np.arange(64) % 20).astype(np.int32))
    assert L.samsim_b200_update_forcing_records(h, 1, 8, None) == -1
    assert L.samsim_b200_update_forcing_records(h, 1, 0, api._dp(buf)) == -1
    assert L.samsim_b200_update_forcing_records(h, 0, 8, api._dp(buf)) == -1
    assert L.samsim_b200_update_forcing_records(h, NREC - 6, 8, api._dp(buf)) == -1
    assert L.samsim_b200_update_forcing_records(h, NREC - 7, 8, api._dp(buf)) == 0
    assert L.samsim_b200_update_forcing_records(h, 1, 8, api._dp(buf)) == 0
    eng.synchronize()


def test_set_forcing_accepts_any_number_of_sites():
    st = scenarios.sheba_state(200)
    ncol = 512
    r0 = 1590   # 16 records around the state's time_counter (1594) keep the 100,000-site table at 51 MB
    eng = _engine(st, ncol, rec_shift=r0)
    rng = np.random.default_rng(14)
    for nsite in (17, 100_000):
        table = _shifted_sites(min(nsite, 1000), 15)[:, :, r0:r0 + 16]
        table = table[rng.integers(0, len(table), nsite)]
        eng.set_forcing(table, rng.integers(0, nsite, ncol).astype(np.int32))
        eng.step(20)
    assert (eng.status() == 0).all()
    table = _era_sites()[:, :, r0:r0 + 16]
    with pytest.raises(api.SamsimError) as e:
        eng.set_forcing(table, np.full(ncol, 9, dtype=np.int32))
    assert e.value.code == -1
    with pytest.raises(api.SamsimError) as e:
        eng.set_forcing(table[:0])
    assert e.value.code == -1
    s = np.ascontiguousarray(table)
    assert eng.L.samsim_b200_set_forcing(eng.h, -3, 16, api._dp(s), None, None, None) == -1
    eng.step(20)   # the rejected calls left the last table in place
    assert (eng.status() == 0).all()


@pytest.mark.skipif(os.environ.get("SAMSIM_SLOW") != "1", reason="17.8 GB forcing table; set SAMSIM_SLOW=1")
def test_site_index_past_2_31_elements():
    st = scenarios.sheba_state(200)
    nsite = 190_000
    sites = np.array([3, 184_001, 187_654, 189_999], dtype=np.int32)   # (site*4 + kind)*NREC >= 2^31 above 183,400
    era = _era_sites()
    table = np.zeros((nsite, 4, NREC))   # untouched pages cost no host memory
    for q, s in enumerate(sites):
        table[s] = era[q + 1] * (1.0 + 0.01 * q)
    big = _engine(st, len(sites))
    big.set_forcing(table, sites)
    del table
    big.step(3000)
    for q, s in enumerate(sites):
        one = _engine(st, 1)
        one.set_forcing(era[q + 1] * (1.0 + 0.01 * q))
        one.step(3000)
        for name in pu.CMP_ARRAYS:
            assert pu.same_bits(big.get_array(name, q, 1), one.get_array(name)).all(), (s, name)
        for name in api.SCALAR_IDS:
            assert pu.same_bits(big.get_scalar(name, q, 1), one.get_scalar(name)).all(), (s, name)
        assert np.array_equal(big.get_int("N_active", q, 1), one.get_int("N_active"))
        assert int(big.get_int("status", q, 1)[0]) == 0
