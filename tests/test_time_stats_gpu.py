"""Per-column time statistics over windows of output records (samsim_b200_set_time_stats), on the GPU, bit for bit
against a numpy implementation of the contract in include/samsim_b200.h fed from step-by-record snapshots."""
import sys
from pathlib import Path

import numpy as np
import pytest

from samsim_b200 import api
from oracle import parity_util as pu

sys.path.insert(0, str(Path(__file__).resolve().parent))
import scenarios  # noqa: E402
from time_stats_ref import STATS, reference  # noqa: E402

pytestmark = pytest.mark.gpu

NCOL = 3000
IOUT = 99                 # a record every 100 steps: 1,000 steps write 10 records
HALF = 500                # the run is driven in two halves; between them (after record 5) some columns fail
RPW = 3                   # windows of records {1,2,3} {4,5,6} {7,8,9}, then {10} closed by hand
WINDOWS = [[0, 1, 2], [3, 4, 5], [6, 7, 8], [9]]
DEPTHS = np.linspace(0.02, 2.5, 25)   # the ice is about 1.5 m thick: the deepest depths lie below every column
PROFILES = ("T", "S_bu", "psi_l")
SUBSET = ["thick_snow", "T_snow", "thickness", "T_top", "N_active"]   # not in id order on purpose
NSC = len(api.SNAP_SCALARS)


# ---- set-up ------------------------------------------------------------------------------------------------------
def _perturbations(ncol, seed):
    rng = np.random.default_rng(seed)
    scale = np.ones((4, ncol))
    offset = np.zeros((4, ncol))
    scale[0], scale[1], scale[3] = rng.uniform(0.8, 1.2, ncol), rng.uniform(0.95, 1.05, ncol), rng.uniform(0.5, 1.5, ncol)
    offset[2] = rng.uniform(-3, 3, ncol)
    return scale, offset


THIN = ((1000, 500), (2500, 300))
SCALE, OFFSET = _perturbations(NCOL, 11)
_rng = np.random.default_rng(12)
FAILED = _rng.choice(NCOL, 40, replace=False)                                  # status 99 before the run
ENDS = _rng.choice(np.setdiff1d(np.arange(NCOL), FAILED), 60, replace=False)
KILLED = _rng.choice(np.setdiff1d(np.arange(NCOL), np.concatenate([FAILED, ENDS])), 5, replace=False)  # after record 5
STEADY = np.setdiff1d(np.arange(NCOL), np.concatenate([FAILED, ENDS, KILLED]))[0]   # contributes every record


def _engine(two_pass=False, ncol=NCOL, i_time_out=IOUT, n_time_out=0):
    st = scenarios.sheba_state(200)
    cfg = api.Config.from_state(st)
    cfg.i_time_out = i_time_out
    eng = api.Engine(cfg, ncol)
    eng.load_column_state(st, 0, set_clock=False)
    eng.broadcast_column(0, 0, ncol)
    if ncol == NCOL:   # two blocks of columns start from the thinner ice of early November (0.46 m, 46 layers)
        thin = scenarios.sheba_state(100)
        for c0, n in THIN:
            eng.load_column_state(thin, c0, set_clock=False)
            eng.broadcast_column(c0, c0 + 1, n - 1)
    eng.set_clock(st["time"], st["i"], n_time_out, st["time_counter"])
    scale, offset = (SCALE, OFFSET) if ncol == NCOL else _perturbations(ncol, ncol)
    eng.set_forcing(scenarios.sheba_forcing(), None, scale, offset)
    eng.set_tuning(two_pass)
    eng.set_snapshot_mode(api.SNAP_FULL)
    return eng, st


def _end_steps(i0):
    end = np.full(NCOL, np.iinfo(np.int64).max, dtype=np.int64)
    end[ENDS[:15]] = i0 + 150     # inside window 1, between records 1 and 2
    end[ENDS[15:30]] = i0 + 400   # on record 4: counted there, excluded from record 5 on
    end[ENDS[30:45]] = i0 + 750   # inside window 3, between records 7 and 8
    end[ENDS[45:]] = i0 + 7       # before the first record
    return end


def _prepare(eng, st):
    status = eng.status()
    status[FAILED] = 99
    eng.set_int("status", status)
    end = _end_steps(st["i"])
    eng.set_end_step(end)
    return end


def _kill(eng):
    status = eng.status()
    status[KILLED] = 99
    eng.set_int("status", status)


def _drive(eng, before=(HALF,), after=(HALF,), close=True):
    for n in before:
        eng.step(n)
    _kill(eng)
    for n in after:
        eng.step(n)
    if close:
        eng.close_time_window()


def _snapshot(eng, names=("thick",) + PROFILES, col0=0, n=None, block=8192):
    n = eng.ncol - col0 if n is None else n
    out = {k: [] for k in api.SNAP_SCALARS + list(names)}
    for c0 in range(col0, col0 + n, block):
        s = eng.get_snapshot(c0, min(block, col0 + n - c0))
        for k in out:
            out[k].append(s[k])
    return {k: np.concatenate(v) for k, v in out.items()}


def _all_state(eng):
    d = {n: eng.get_array(n) for n in pu.CMP_ARRAYS}
    d.update({n: eng.get_scalar(n) for n in api.SCALAR_IDS})
    d.update({n: eng.get_int(n) for n in api.INT_IDS})
    d.update({"clock_" + k: np.float64(v) for k, v in eng.get_clock().items()})
    return d


def _differ(a, b):
    return [n for n in a if not pu.same_bits(a[n], b[n]).all()]


def _hist_equal(h1, h2, keys=("nrec", "i_first", "i_last")):
    for k in keys:
        assert np.array_equal(h1[k], h2[k]), k
    assert pu.same_bits(h1["time_first"], h2["time_first"]).all() and pu.same_bits(h1["time_last"], h2["time_last"]).all()
    assert h1["quantities"] == h2["quantities"]
    for k in STATS:
        assert h1[k].shape == h2[k].shape, k
        bad = ~pu.same_bits(h1[k], h2[k])
        assert not bad.any(), (k, np.argwhere(bad)[:5])


def _matches_reference(hist, ref):
    for s, k in enumerate(STATS):
        bad = ~pu.same_bits(hist[k], ref[..., s])
        assert not bad.any(), (k, np.argwhere(bad)[:5], hist[k][bad][:5], ref[..., s][bad][:5])


@pytest.fixture(scope="module")
def run():
    """A: all scalars and three profiles, B: a scalar subset, both driven in two multi-record calls; R: steps to each
    record and keeps snapshot, status and end steps; P: the same run without statistics"""
    a, st = _engine()
    b, _ = _engine()
    r, _ = _engine()
    p, _ = _engine()
    end = None
    for eng in (a, b, r, p):
        end = _prepare(eng, st)
    a.set_time_stats(RPW, None, DEPTHS, PROFILES, max_windows=8)
    b.set_time_stats(RPW, SUBSET, max_windows=8)
    for eng in (a, b):
        _drive(eng)
    _drive(p, close=False)
    recs, left = [], 2 * HALF
    while left > 0:
        n = min(r.steps_to_next_output(), left)
        r.step(n)
        left -= n
        if r.get_clock()["n_time_out"] == 0:
            recs.append((r.get_clock()["i"], _snapshot(r), r.status(), end))
        if left == HALF:
            _kill(r)
    return a, b, r, p, st, recs, a.time_stats(), b.time_stats()


def test_history_matches_the_numpy_reference(run):
    a, b, r, p, st, recs, ha, hb = run
    assert len(recs) == 10 and a.time_stats_held() == 4 and b.time_stats_held() == 4
    assert list(ha["nrec"]) == [3, 3, 3, 1]
    ri = [i for i, *_ in recs]
    assert list(ha["i_first"]) == [ri[w[0]] for w in WINDOWS] and list(ha["i_last"]) == [ri[w[-1]] for w in WINDOWS]
    t = [s["time"][STEADY] for _, s, _, _ in recs]
    assert pu.same_bits(ha["time_first"], [t[w[0]] for w in WINDOWS]).all()
    assert pu.same_bits(ha["time_last"], [t[w[-1]] for w in WINDOWS]).all()
    assert ha["quantities"][:NSC] == [(n, None) for n in api.SNAP_SCALARS]
    assert ha["quantities"][NSC] == ("T", DEPTHS[0]) and len(ha["quantities"]) == NSC + 3 * len(DEPTHS)
    assert hb["quantities"] == [(n, None) for n in api.SNAP_SCALARS if n in SUBSET]
    _matches_reference(ha, reference(recs, WINDOWS, depths=DEPTHS, profiles=PROFILES))
    _matches_reference(hb, reference(recs, WINDOWS, scalars=SUBSET))
    idx = [api.SNAP_SCALARS.index(q) for q, _ in hb["quantities"]]   # each quantity is accumulated on its own
    _hist_equal(hb, {**ha, **{k: ha[k][..., idx] for k in STATS}, "quantities": hb["quantities"]})

    cnt = ha["count"]
    assert (cnt[:, FAILED] == 0).all() and np.isnan(ha["mean"][:, FAILED]).all() and np.isnan(ha["max"][:, FAILED]).all()
    assert (cnt[:, STEADY, :NSC] == ha["nrec"][:, None]).all()
    assert (cnt[:, STEADY, -1] == 0).all() and np.isnan(ha["var"][:, STEADY, -1]).all()   # the deepest depth
    prof = cnt[:, :, NSC:]
    assert (prof == 0).any() and (prof > 0).any()
    # a column that fails between two records of a window keeps the records it contributed before
    assert (cnt[1, KILLED, :NSC] == 2).all() and (cnt[2:, KILLED] == 0).all()
    # end steps inside windows
    e = ENDS
    assert (cnt[0, e[:15], 0] == 1).all() and (cnt[1:, e[:15], 0] == 0).all()
    assert (cnt[1, e[15:30], 0] == 1).all() and (cnt[0, e[15:30], 0] == 3).all() and (cnt[2:, e[15:30], 0] == 0).all()
    assert (cnt[2, e[30:45], 0] == 1).all() and (cnt[3, e[30:45], 0] == 0).all()
    assert (cnt[:, e[45:]] == 0).all()
    assert (ha["var"][:3, STEADY, :NSC] > 0).any(axis=-1).all()   # the records differ


def test_stepping_is_unchanged(run):
    a, b, r, p, st, recs, ha, hb = run
    sa, sb, sr, sp = _all_state(a), _all_state(b), _all_state(r), _all_state(p)
    for other in (sb, sr, sp):
        assert not _differ(sa, other), _differ(sa, other)
    assert p.launch_count() <= a.launch_count() <= p.launch_count() + len(recs)


@pytest.mark.parametrize("variant", ["two_pass", "rebinned", "uneven", "with_group_stats"])
def test_history_does_not_depend_on_order(run, variant):
    ha = run[6]
    e, st = _engine(two_pass=(variant == "two_pass"))
    _prepare(e, st)
    if variant == "rebinned":
        assert e.rebin()   # the failed columns move to the end
        e.set_rebin_interval(70)
    goc = (np.arange(NCOL) % 7).astype(np.int32)
    if variant == "with_group_stats":
        e.set_group_stats(goc, DEPTHS, PROFILES, max_records=16)
    e.set_time_stats(RPW, None, DEPTHS, PROFILES, max_windows=8)
    if variant == "uneven":   # single steps, short calls, calls across several records and windows
        _drive(e, (1, 7, 250, 99, 143), (7, 1, 300, 192))
    else:
        _drive(e)
    if variant == "rebinned":
        assert e.divergence()["rebins"] >= 2
    _hist_equal(e.time_stats(clear=True), ha)
    assert e.time_stats_held() == 0
    if variant == "with_group_stats":   # and the group statistics equal those of a run without time statistics
        g, _ = _engine()
        _prepare(g, st)
        g.set_group_stats(goc, DEPTHS, PROFILES, max_records=16)
        _drive(g, close=False)
        h1, h2 = e.group_stats(), g.group_stats()
        assert np.array_equal(h1["i"], h2["i"]) and pu.same_bits(h1["time"], h2["time"]).all()
        for k in STATS:
            assert pu.same_bits(h1[k], h2[k]).all(), k


# ---- window rules, arguments ---------------------------------------------------------------------------------------
def _small(ncol=256):
    return _engine(ncol=ncol, i_time_out=9)   # a record every 10 steps


def _record(eng, recs):
    eng.step(eng.steps_to_next_output())
    recs.append((eng.get_clock()["i"], _snapshot(eng, ("thick", "T")), eng.status(),
                 np.full(eng.ncol, np.iinfo(np.int64).max)))


def test_manual_windows_of_different_lengths():
    e, st = _small()
    L, hd = e.L, e.h
    e.set_time_stats(0, None, DEPTHS[:5], ("T",), max_windows=3)
    assert L.samsim_b200_close_time_window(hd) == -5      # nothing recorded yet
    recs = []
    for _ in range(2):
        _record(e, recs)
    e.close_time_window()
    assert L.samsim_b200_close_time_window(hd) == -5      # the new window is empty
    for _ in range(3):
        _record(e, recs)
    e.step(4)                                             # steps without a record do not count
    e.close_time_window()
    h = e.time_stats()
    assert list(h["nrec"]) == [2, 3] and list(h["i_last"]) == [recs[1][0], recs[4][0]]
    _matches_reference(h, reference(recs, [[0, 1], [2, 3, 4]], depths=DEPTHS[:5], profiles=("T",)))
    e.step(1000)                                          # records_per_window = 0: stepping completes no window
    assert e.time_stats_held() == 2
    e.close_time_window()
    assert e.time_stats_held() == 3 and e.time_stats()["nrec"][2] == 100
    e.step(10)
    assert L.samsim_b200_close_time_window(hd) == -5      # the history is full


def test_capacity_clear_and_new_setting():
    e, st = _small()
    L, hd = e.L, e.h
    e.set_time_stats(1, ["thickness"], max_windows=2)
    e.step(20)
    assert e.time_stats_held() == 2
    clk, launches, th = e.get_clock(), e.launch_count(), e.get_array("thick")
    assert L.samsim_b200_step(hd, 10) == -5 and L.samsim_b200_step(hd, 1000) == -5
    assert e.get_clock() == clk and e.launch_count() == launches and pu.same_bits(e.get_array("thick"), th).all()
    e.step(9)                                             # up to, not onto, the next record
    assert e.time_stats_held() == 2
    # records_per_window = 2, one window of room: the record that would complete a second one is refused
    e.set_time_stats(2, ["thickness"], max_windows=1)
    assert e.time_stats_held() == 0
    e.step(1 + 10)                                        # records 1 and 2: one window
    assert e.time_stats_held() == 1
    e.step(10)                                            # record 3 opens the next window
    assert L.samsim_b200_step(hd, 10) == -5
    # clear drops the held windows only: the window in progress keeps record 3
    i3 = e.get_clock()["i"]
    e.clear_time_stats()
    assert e.time_stats_held() == 0
    e.step(10)
    h = e.time_stats()
    assert list(h["nrec"]) == [2] and list(h["i_first"]) == [i3] and list(h["i_last"]) == [i3 + 10]
    # a new setting drops the held windows and the window in progress
    e.step(10)
    e.set_time_stats(2, ["thickness"], max_windows=4)
    assert e.time_stats_held() == 0
    i0 = e.get_clock()["i"]
    e.step(20)
    h = e.time_stats()
    assert list(h["i_first"]) == [i0 + 10] and list(h["i_last"]) == [i0 + 20]


def test_arguments_and_snapshot_mode():
    e, st = _small()
    L, hd = e.L, e.h
    z = np.ascontiguousarray(DEPTHS)
    ALL = (1 << NSC) - 1

    def setts(rpw=3, scm=ALL, nz=3, depth=z, mask=1, mx=2):
        return L.samsim_b200_set_time_stats(hd, rpw, scm, nz, api._dp(depth) if depth is not None else None, mask, mx)

    assert setts() == 0
    # every bad argument: SAMSIM_ERR_ARG and the previous setting stays
    assert setts(rpw=-1) == -1 and setts(mx=0) == -1 and setts(scm=1 << NSC) == -1
    assert setts(depth=np.array([0.1, 0.1, 0.2])) == -1
    assert setts(depth=np.array([0.0, 0.1, 0.2])) == -1
    assert setts(depth=np.array([0.3, 0.2, 0.4])) == -1
    assert setts(depth=np.array([0.1, np.inf, 0.4])) == -1
    assert setts(depth=np.array([0.1, np.nan, 0.4])) == -1
    assert setts(depth=np.array([-0.1, 0.1, 0.4])) == -1
    assert setts(depth=None) == -1 and setts(nz=-1) == -1
    assert setts(mask=1 << api.SNAP_ARRAYS.index("ray")) == -1
    assert setts(mask=1 << api.SNAP_ARRAYS.index("bgc1_bu")) == -1   # N_bgc = 0
    assert setts(mask=1 << 14) == -1
    assert setts(nz=0, mask=1) == -1
    assert L.samsim_b200_set_time_stats(None, 1, 1, 0, None, 0, 1) == -1
    assert L.samsim_b200_time_stats_held(None) == -1
    assert L.samsim_b200_close_time_window(None) == -1 and L.samsim_b200_clear_time_stats(None) == -1
    assert L.samsim_b200_get_time_stats(None, None, None, None, None, 0, 0, 0, 0) == -1
    # the first setting is still in place: profiles (FULL needed) and windows of three records
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_SCALARS_ONLY) == -5
    e.step(20)
    assert e.time_stats_held() == 0
    e.step(10)
    assert e.time_stats_held() == 1
    # get: range checks
    Q = NSC + 3
    buf = np.empty(2 * 4 * Q * 5)
    assert L.samsim_b200_get_time_stats(hd, api._dp(buf), None, None, None, 0, 2, 0, 4) == -1   # one window held
    assert L.samsim_b200_get_time_stats(hd, api._dp(buf), None, None, None, -1, 1, 0, 4) == -1
    assert L.samsim_b200_get_time_stats(hd, api._dp(buf), None, None, None, 0, -1, 0, 4) == -1
    assert L.samsim_b200_get_time_stats(hd, api._dp(buf), None, None, None, 0, 1, -1, 4) == -1
    assert L.samsim_b200_get_time_stats(hd, api._dp(buf), None, None, None, 0, 1, 0, -1) == -1
    assert L.samsim_b200_get_time_stats(hd, api._dp(buf), None, None, None, 0, 1, 253, 4) == -1
    assert L.samsim_b200_get_time_stats(hd, api._dp(buf), None, None, None, 0, 1, 252, 4) == 0
    assert L.samsim_b200_get_time_stats(hd, None, None, None, None, 0, 1, 0, 256) == 0
    # the snapshot mode
    assert setts(mask=0) == 0                                            # scalars only: SCALARS is enough
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_SCALARS_ONLY) == 0
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_NONE) == -5
    assert setts() == -5                                                 # FULL needed
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_SCALARS_ONLY) == 0   # the scalar setting stays
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_NONE) == -5
    assert setts(scm=0, mask=0) == 0 and e.time_stats_held() == 0      # off
    assert L.samsim_b200_close_time_window(hd) == -5
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_NONE) == 0
    assert setts(mask=0) == -5
    assert setts(scm=0, mask=1) == -5


def test_large_batch_crosses_2_31_history_elements():
    """1,048,576 columns, Q = 120, one window per record, a record at every step: 4 windows of 6.3e8 doubles"""
    ncol = 1 << 20
    depths = np.linspace(0.04, 2.0, 50)
    e, st = _engine(ncol=ncol, i_time_out=0)
    e.set_time_stats(1, None, depths, ("T", "S_bu"), max_windows=4)
    rng = np.random.default_rng(13)
    sample = [(int(c), 1) for c in np.sort(rng.choice(ncol - 1024, 48, replace=False))] + [(ncol - 1024, 1024)]
    recs = {s: [] for s in sample}
    end = np.full(ncol, np.iinfo(np.int64).max)
    for _ in range(4):
        e.step(1)
        i, status = e.get_clock()["i"], e.status()
        for c0, n in sample:
            recs[(c0, n)].append((i, _snapshot(e, ("thick", "T", "S_bu"), c0, n), status[c0:c0 + n], end[c0:c0 + n]))
    assert e.time_stats_held() == 4
    Q = NSC + 2 * len(depths)
    assert 4 * ncol * Q * 5 > 2 ** 31
    for (c0, n), rr in recs.items():
        h = e.time_stats(c0, n)
        assert h["count"].shape == (4, n, Q) and list(h["nrec"]) == [1] * 4
        assert list(h["i_first"]) == [i for i, *_ in rr] and list(h["i_last"]) == list(h["i_first"])
        _matches_reference(h, reference(rr, [[0], [1], [2], [3]], depths=depths, profiles=("T", "S_bu")))
    assert (h["count"][:, :, :NSC] == 1).all() and (h["var"][:, :, :NSC] == 0).all()
