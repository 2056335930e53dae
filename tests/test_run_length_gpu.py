"""Runs of different lengths in one batch: per-column end steps (samsim_b200_set_end_step), per-set lab lengths
(samsim_b200_set_lab_lengths) and the batch driver samsim_grotz_batch, on the GPU against the oracle and against
runs of one column each."""
import sys
from pathlib import Path

import numpy as np
import pytest

from samsim_b200 import api
from oracle import parity_util as pu

sys.path.insert(0, str(Path(__file__).resolve().parent))
import scenarios  # noqa: E402

pytestmark = pytest.mark.gpu

NO_END = np.iinfo(np.int64).max


def _fmt(bad, n=12):
    return "\n".join(bad[:n]) + (f"\n... {len(bad)} mismatches" if len(bad) > n else "")


def _state(eng, col):
    """every array, scalar and int of one engine column"""
    d = {n: eng.get_array(n, col, 1)[0] for n in pu.CMP_ARRAYS}
    d.update({n: eng.get_scalar(n, col, 1)[:1] for n in api.SCALAR_IDS})
    d.update({n: eng.get_int(n, col, 1)[:1] for n in api.INT_IDS})
    return d


def _changed(a, b):
    return [n for n in a if not pu.same_bits(a[n], b[n]).all()]


def _lab_sets(n, nset):
    base = scenarios.lab_series(n)
    return np.stack([base * np.array([1.0 + 0.03 * q, 1.0 + 0.5 * q, 1.0, 1.0])[:, None] for q in range(nset)])


# testcases 101-105 and 101 again without an end; 3602 is an output step (records at i = 1 + k*3601)
LAB_TCS = [101, 102, 103, 104, 105, 101]
LAB_ENDS = [2000, 3601, 3602, 9000, 14000, None]
LAB_TOTAL = 20000


@pytest.fixture(scope="module")
def lab_oracles(oracle_mod):
    """oracle columns advanced exactly their own number of steps, with their output records"""
    sets = _lab_sets(LAB_TOTAL, len(LAB_TCS))
    lens = [e if e is not None else LAB_TOTAL for e in LAB_ENDS]
    fresh, done = [], []
    for q, tc in enumerate(LAB_TCS):
        col = oracle_mod.Column(tc, "det")
        col.set_lab_forcing(*sets[q][:, :lens[q]])
        fresh.append((col.state(), col.scalar("S_total")))
        col.record_outputs()
        assert col.step(lens[q]) == 0
        done.append(col)
    return sets, lens, fresh, done


@pytest.mark.parametrize("two_pass", [False, True])
def test_columns_stop_at_their_own_end_step(oracle_mod, lab_oracles, two_pass):
    sets, lens, fresh, cols = lab_oracles
    n = len(LAB_TCS)
    eng = api.Engine(pu.config_from_oracle(cols[0]), n)
    eng.set_tuning(two_pass)
    for q, (st, S_total) in enumerate(fresh):
        eng.load_column_state(st, q, set_clock=(q == 0))
        eng.set_scalar("S_total", [S_total], col0=q)
    # each set holds exactly the records its column reads; NaN behind them would show any read past the end
    table = np.full((n, 4, LAB_TOTAL), np.nan)
    for q in range(n):
        table[q, :, :lens[q]] = sets[q][:, :lens[q]]
    eng.set_lab_forcing(table, np.arange(n, dtype=np.int32), nrec_of_set=lens)
    eng.set_end_step([e for e in LAB_ENDS[:5]])  # column 5 keeps the default: no end
    eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    eng.clear_events()

    eng.step(5000)    # column 0 ends inside this launch
    first = _state(eng, 0)
    eng.step(15000)   # the others end inside this one
    assert eng.get_clock()["i"] == LAB_TOTAL
    assert not _changed(first, _state(eng, 0)), "a finished column changed"
    assert (eng.status() == 0).all()
    snap = eng.get_snapshot(arrays=False)
    for q, col in enumerate(cols):
        # the clock is batch-wide: the column matches the oracle in everything but the clock
        bad = [b for b in pu.compare_column(col, eng, q, label=f"testcase {LAB_TCS[q]} end {lens[q]}: ") if "clock" not in b]
        assert not bad, _fmt(bad)
        o, g = col.events(), eng.events(q)
        assert o == g - scenarios.DEVICE_ONLY, (q, sorted(o ^ g))
        rec = col.records[-1]   # the last record at or before the column's end
        for name in oracle_mod.SNAP_SCALARS:
            assert pu.same_bits(snap[name][q], rec[name]), (q, name, snap[name][q], rec[name])
        assert snap["N_active"][q] == rec["N_active"]
    assert [int(c.records[-1]["time"]) for c in cols] == [0, 0, 3601, 7202, 10803, 18005]
    assert max(c.int("N_active") for c in cols) >= 3


def _tc1_ensemble(oracle_mod, ncol, ends):
    base = oracle_mod.Column(1, "det")
    eng = pu.engine_from_oracle(base, ncol=ncol)
    rng = np.random.default_rng(7)
    Sb = 34.0 + rng.normal(0, 0.5, ncol)
    Tb = np.maximum(-1.0 + rng.normal(0, 0.05, ncol), -1.7)
    m1 = base.array("m")[0]
    eng.set_scalar("T_top", -5.0 + rng.normal(0, 0.5, ncol))
    eng.set_scalar("T_bottom", Tb)
    eng.set_scalar("S_bu_bottom", Sb)
    eng.set_scalar("fl_q_bottom", np.abs(rng.normal(0, 2.0, ncol)))
    S = np.tile(base.array("S_abs"), (ncol, 1)); S[:, 0] = Sb * m1; eng.set_array("S_abs", S)
    H = np.tile(base.array("H_abs"), (ncol, 1)); H[:, 0] = m1 * Tb * 3400.0; eng.set_array("H_abs", H)
    eng.set_array("T", np.repeat(Tb[:, None], 90, 1)); eng.set_array("S_bu", np.repeat(Sb[:, None], 90, 1))
    eng.set_end_step(ends)
    return eng


def test_end_steps_survive_rebinning(oracle_mod):
    ncol = 384
    rng = np.random.default_rng(3)
    ends = rng.choice(np.array([700, 1500, 2600, 3900, NO_END], dtype=np.int64), ncol)
    moved = rng.choice(ncol, 40, replace=False)
    a, b = _tc1_ensemble(oracle_mod, ncol, ends), _tc1_ensemble(oracle_mod, ncol, ends)
    for eng in (a, b):
        eng.step(2000)
    at2000 = {n: b.get_array(n) for n in pu.CMP_ARRAYS}
    assert a.rebin()
    slot = a.slot_map()
    done = ends <= 2000
    assert slot[done].min() > slot[~done].max()   # finished columns sit last, with the failed ones
    for eng in (a, b):     # end steps set after re-binning go through the slot map
        for c in moved:
            eng.set_end_step([2400 if ends[c] > 2400 else ends[c]], col0=int(c))
    a.set_rebin_auto(1e-6)
    for eng in (a, b):
        eng.step(1500)
        eng.step(1500)
    assert a.divergence()["rebins"] >= 1 and b.divergence()["rebins"] == 0
    assert (a.status() == 0).all() and (b.status() == 0).all()
    for name in pu.CMP_ARRAYS:
        assert pu.same_bits(a.get_array(name), b.get_array(name)).all(), name
    for name in api.SCALAR_IDS:
        assert pu.same_bits(a.get_scalar(name), b.get_scalar(name)).all(), name
    for name in api.INT_IDS:
        assert np.array_equal(a.get_int(name), b.get_int(name)), name
    for name in pu.CMP_ARRAYS:   # the columns that had ended by step 2000 did not move since
        assert pu.same_bits(at2000[name][done], a.get_array(name)[done]).all(), name
    live = a.get_array("T")[ends == NO_END]
    assert not pu.same_bits(at2000["T"][ends == NO_END], live).all()


def _lab_engine(oracle_mod, nrec, lengths=None):
    cols = [oracle_mod.Column(tc, "det") for tc in (101, 102)]
    eng = api.Engine(pu.config_from_oracle(cols[0]), 2)
    for q, col in enumerate(cols):
        eng.load_column_state(col.state(), q, set_clock=(q == 0))
        eng.set_scalar("S_total", [col.scalar("S_total")], col0=q)
    eng.set_lab_forcing(_lab_sets(nrec, 2), np.arange(2, dtype=np.int32), nrec_of_set=lengths)
    return eng


def test_lab_lengths_are_enforced(oracle_mod):
    # column 1 runs on, but its set ends at record 3000: the call stops there
    eng = _lab_engine(oracle_mod, 6000, lengths=[6000, 3000])
    with pytest.raises(api.SamsimError) as e:
        eng.step(5000)
    assert e.value.code == -5 and eng.get_clock()["i"] == 3000
    with pytest.raises(api.SamsimError):
        eng.step(1)
    assert eng.get_clock()["i"] == 3000
    # once the column ends within its set, the batch runs on; column 0's set bounds the run
    eng.set_end_step([3000], col0=1)
    frozen = _state(eng, 1)
    eng.step(2000)
    assert not _changed(frozen, _state(eng, 1))
    eng.step(1000)
    with pytest.raises(api.SamsimError) as e:
        eng.step(10)
    assert e.value.code == -5 and eng.get_clock()["i"] == 6000
    # a set whose columns have all finished does not bound the run
    eng.set_end_step([6000], col0=0)
    eng.step(10)
    assert eng.get_clock()["i"] == 6010 and (eng.status() == 0).all()
    # without set_lab_lengths every set holds nrec records, the single bound of before
    eng = _lab_engine(oracle_mod, 3000)
    with pytest.raises(api.SamsimError) as e:
        eng.step(5000)
    assert e.value.code == -5 and eng.get_clock()["i"] == 3000


def test_grotz_batch_equals_single_runs(tmp_path):
    from samsim_b200 import grotz
    tcs = [101, 102, 103, 104, 105]
    max_steps = [2 * 3601 + 1, 3601 + 1, 3 * 3601 + 1, 4 * 3601 + 1, 2 * 3601 + 500]
    labdir = tmp_path / "2017_input"
    labdir.mkdir()
    head = 20000   # more than any member reads; the rest pads the files to length_input_lab
    for q, tc in enumerate(tcs):
        nrec = grotz.init_testcase(tc)["length_input_lab"]
        series = scenarios.lab_series(head, styropor_hours=(1, 2)) * np.array([1.0 + 0.03 * q, 1.0 + 0.5 * q, 1.0, 1.0])[:, None]
        for name, row in zip(["Tice", "snowfall", "heat", "styropor"], series):
            path = labdir / f"{name}_exp_{tc - 100}.txt"
            np.savetxt(path, row, fmt="%.9e")
            with open(path, "a") as f:
                f.write("0\n" * (nrec - head))
    members = [{"testcase": tc, "description": f"lab {tc}", "output_dir": tmp_path / "batch" / str(tc), "max_steps": m}
               for tc, m in zip(tcs, max_steps)]
    assert grotz.grotz_batch(members, lab_input_dir=labdir) == [0] * 5
    for m in members:
        alone = tmp_path / "alone" / str(m["testcase"])
        assert grotz.grotz(m["testcase"], m["description"], output_dir=alone, lab_input_dir=labdir, max_steps=m["max_steps"]) == 0
        names = sorted(p.name for p in alone.glob("dat_*.dat"))
        assert names == sorted(p.name for p in Path(m["output_dir"]).glob("dat_*.dat")) and len(names) == 17
        for name in names:
            mine, ref = (Path(m["output_dir"]) / name).read_bytes(), (alone / name).read_bytes()
            if name == "dat_settings.dat":
                mine, ref = (b"\n".join(ln for ln in x.split(b"\n") if not ln.startswith(b" ncol")) for x in (mine, ref))
            assert mine == ref, (m["testcase"], name)
        nrec = len((alone / "dat_thick.dat").read_text().splitlines())
        assert nrec == (m["max_steps"] - 1) // 3601 + 1
