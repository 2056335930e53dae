"""Ensemble statistics per column group at every output record (samsim_b200_set_group_stats), on the GPU, bit for bit
against a numpy implementation of the contract in include/samsim_b200.h fed from step-by-record snapshots."""
import sys
from pathlib import Path

import numpy as np
import pytest

from samsim_b200 import api
from oracle import parity_util as pu

sys.path.insert(0, str(Path(__file__).resolve().parent))
import scenarios  # noqa: E402
from group_stats_ref import NSC, reference_record  # noqa: E402

pytestmark = pytest.mark.gpu

NCOL = 3000
IOUT = 99                 # a record every 100 steps: 420 steps write 4 records
NSTEP = 420
DEPTHS = np.linspace(0.02, 2.5, 25)   # the ice is about 1.5 m thick: the deepest depths lie below every member
PROFILES = ("T", "S_bu", "psi_l")


# ---- set-up ------------------------------------------------------------------------------------------------------
def _perturbations(ncol, seed):
    rng = np.random.default_rng(seed)
    scale = np.ones((4, ncol))
    offset = np.zeros((4, ncol))
    scale[0], scale[1], scale[3] = rng.uniform(0.8, 1.2, ncol), rng.uniform(0.95, 1.05, ncol), rng.uniform(0.5, 1.5, ncol)
    offset[2] = rng.uniform(-3, 3, ncol)
    return scale, offset


def _groups(ncol, seed):
    """one member, 1,300 members, groups of 15..25, one empty group (the last) and 100 columns in no group"""
    rng = np.random.default_rng(seed)
    perm = rng.permutation(ncol)
    goc = np.full(ncol, -1, dtype=np.int32)
    goc[perm[0]] = 0
    goc[perm[1:1301]] = 1
    rest = perm[1301:ncol - 100]
    g, k = 2, 0
    while k < len(rest):
        n = int(rng.integers(15, 26))
        goc[rest[k:k + n]] = g
        g, k = g + 1, k + n
    return goc, g + 1


THIN = ((1000, 500), (2500, 300))
SCALE, OFFSET = _perturbations(NCOL, 1)
GOC, NGROUP = _groups(NCOL, 2)
_rng = np.random.default_rng(3)
FAILED = _rng.choice(NCOL, 40, replace=False)                 # status 99 before the run
ENDS = _rng.choice(np.setdiff1d(np.arange(NCOL), FAILED), 60, replace=False)


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
    end[ENDS[:20]] = i0 + 150     # between the first and the second record
    end[ENDS[20:40]] = i0 + 300   # on the third record: counted there, excluded from the fourth
    end[ENDS[40:]] = i0 + 7       # before the first
    return end


def _prepare(eng, st):
    status = eng.status()
    status[FAILED] = 99
    eng.set_int("status", status)
    end = _end_steps(st["i"])
    eng.set_end_step(end)
    return end


def _snapshot(eng, names=("thick",) + PROFILES, block=8192):
    out = {n: [] for n in api.SNAP_SCALARS + list(names)}
    for c0 in range(0, eng.ncol, block):
        s = eng.get_snapshot(c0, min(block, eng.ncol - c0))
        for n in out:
            out[n].append(s[n])
    return {n: np.concatenate(v) for n, v in out.items()}


def _all_state(eng):
    d = {n: eng.get_array(n) for n in pu.CMP_ARRAYS}
    d.update({n: eng.get_scalar(n) for n in api.SCALAR_IDS})
    d.update({n: eng.get_int(n) for n in api.INT_IDS})
    d.update({"clock_" + k: np.float64(v) for k, v in eng.get_clock().items()})
    return d


def _differ(a, b):
    return [n for n in a if not pu.same_bits(a[n], b[n]).all()]


def _hist_equal(h1, h2):
    assert np.array_equal(h1["i"], h2["i"]) and pu.same_bits(h1["time"], h2["time"]).all()
    for k in ("count", "mean", "var", "min", "max"):
        assert h1[k].shape == h2[k].shape, k
        bad = ~pu.same_bits(h1[k], h2[k])
        assert not bad.any(), (k, np.argwhere(bad)[:5])


@pytest.fixture(scope="module")
def run():
    """A: the whole stretch in one call with statistics on; B: steps to each record and keeps snapshot, status and end
    steps; P: the same run without statistics"""
    a, st = _engine()
    b, _ = _engine()
    p, _ = _engine()
    end = None
    for eng in (a, b, p):
        end = _prepare(eng, st)
    a.set_group_stats(GOC, DEPTHS, PROFILES, max_records=8, ngroup=NGROUP)
    a.step(NSTEP)
    p.step(NSTEP)
    recs, left = [], NSTEP
    while left > 0:
        n = min(b.steps_to_next_output(), left)
        b.step(n)
        left -= n
        if b.get_clock()["n_time_out"] == 0:
            recs.append((b.get_clock()["i"], _snapshot(b), b.status()))
    ref = np.stack([reference_record(s, stat, end, i, GOC, NGROUP, DEPTHS, PROFILES) for i, s, stat in recs])
    hist = a.group_stats(clear=False)
    return a, b, p, st, recs, ref, hist


def test_history_matches_the_numpy_reference(run):
    a, b, p, st, recs, ref, hist = run
    assert len(recs) == 4 and a.group_stats_held() == 4
    assert list(hist["i"]) == [i for i, _, _ in recs]
    steady = np.setdiff1d(np.arange(NCOL), np.concatenate([FAILED, ENDS]))[0]   # a column that writes every record
    assert pu.same_bits(hist["time"], [s["time"][steady] for _, s, _ in recs]).all()
    assert hist["quantities"][:NSC] == [(n, None) for n in api.SNAP_SCALARS]
    assert hist["quantities"][NSC] == ("T", DEPTHS[0]) and len(hist["quantities"]) == NSC + 3 * len(DEPTHS)
    for s, k in enumerate(("count", "mean", "var", "min", "max")):
        bad = ~pu.same_bits(hist[k], ref[..., s])
        assert not bad.any(), (k, np.argwhere(bad)[:5], hist[k][bad][:5], ref[..., s][bad][:5])
    cnt = hist["count"]
    assert (cnt[:, 0, 0] <= 1).all()   # one member
    assert (cnt[:, NGROUP - 1] == 0).all() and np.isnan(hist["mean"][:, NGROUP - 1]).all()   # the empty group
    assert cnt[0, 1, 0] > 1024
    prof = cnt[:, :, NSC:]
    assert (prof == 0).any() and ((prof > 0) & (prof < cnt[:, :, :1])).any()   # depths below all and below some ice
    assert (hist["var"][:, 1, :NSC][:, [0, 5, 8]] > 0).all()   # the members differ


def test_stepping_is_unchanged(run):
    a, b, p, st, recs, ref, hist = run
    sa, sb, sp = _all_state(a), _all_state(b), _all_state(p)
    assert not _differ(sa, sb), _differ(sa, sb)
    assert not _differ(sa, sp), _differ(sa, sp)
    assert p.launch_count() <= a.launch_count() <= p.launch_count() + len(recs)


def test_exclusions(run):
    a, b, p, st, recs, ref, hist = run
    i0 = st["i"]
    for r, (i, _, status) in enumerate(recs):
        assert (status[FAILED] == 99).all()
        live = (status == 0) & (_end_steps(i0) >= i)
        for g in range(NGROUP):
            assert hist["count"][r, g, 0] == live[GOC == g].sum()
    # columns whose end step lies between two records are counted before it and not after
    grouped = ENDS[:20][GOC[ENDS[:20]] >= 0]
    assert len(grouped) > 0
    assert (recs[0][2][grouped] == 0).all() and recs[0][0] < i0 + 150 < recs[1][0]


@pytest.mark.parametrize("variant", ["two_pass", "rebinned", "uneven"])
def test_history_does_not_depend_on_order(run, variant):
    hist = run[-1]
    e, st = _engine(two_pass=(variant == "two_pass"))
    _prepare(e, st)
    if variant == "rebinned":
        assert e.rebin()   # the failed columns move to the end
        e.set_rebin_interval(70)
    e.set_group_stats(GOC, DEPTHS, PROFILES, max_records=8, ngroup=NGROUP)
    for n in ((NSTEP,) if variant != "uneven" else (1, 37, 150, 99, 13, 120)):
        e.step(n)
    if variant == "rebinned":
        assert e.divergence()["rebins"] >= 2
    _hist_equal(e.group_stats(), hist)
    assert e.group_stats_held() == 0


def test_one_group_per_column():
    e, st = _engine(ncol=512)
    e.set_group_stats(np.arange(512), DEPTHS[:5], ("T",), max_records=4)
    e.step(250)
    s = _snapshot(e, ("thick", "T"))
    h = e.group_stats()
    assert h["count"].shape == (2, 512, NSC + 5)
    sc = np.stack([s[n] for n in api.SNAP_SCALARS], 1)
    assert pu.same_bits(h["mean"][-1, :, :NSC], sc).all()
    assert (h["count"][-1, :, :NSC] == 1).all() and (h["var"][-1, :, :NSC] == 0).all()
    assert pu.same_bits(h["min"][-1], h["mean"][-1]).all() and pu.same_bits(h["max"][-1], h["mean"][-1]).all()


def test_capacity_and_arguments():
    e, st = _engine(ncol=256)
    L, hd = e.L, e.h
    z = np.ascontiguousarray(DEPTHS)
    goc = np.zeros(256, dtype=np.int32)

    def setgs(ng=2, g=goc, nz=3, depth=z, mask=1, mx=2):
        g = None if g is None else np.ascontiguousarray(g, dtype=np.int32)
        return L.samsim_b200_set_group_stats(hd, ng, api._ip(g), nz, api._dp(depth) if depth is not None else None, mask, mx)

    assert setgs() == 0
    # every bad argument: SAMSIM_ERR_ARG and the previous setting stays
    bad_goc = goc.copy(); bad_goc[7] = 2
    assert setgs(g=bad_goc) == -1
    bad_goc[7] = -2
    assert setgs(g=bad_goc) == -1
    assert setgs(ng=-1) == -1 and setgs(mx=0) == -1
    assert setgs(depth=np.array([0.1, 0.1, 0.2])) == -1
    assert setgs(depth=np.array([0.0, 0.1, 0.2])) == -1
    assert setgs(depth=np.array([0.3, 0.2, 0.4])) == -1
    assert setgs(depth=np.array([0.1, np.inf, 0.4])) == -1
    assert setgs(depth=np.array([-0.1, 0.1, 0.4])) == -1
    assert setgs(depth=None) == -1 and setgs(nz=-1) == -1
    assert setgs(mask=1 << api.SNAP_ARRAYS.index("ray")) == -1
    assert setgs(mask=1 << api.SNAP_ARRAYS.index("bgc1_bu")) == -1   # N_bgc = 0
    assert setgs(mask=1 << 14) == -1
    assert setgs(nz=0, mask=1) == -1
    assert L.samsim_b200_set_group_stats(None, 1, None, 0, None, 0, 1) == -1
    assert L.samsim_b200_group_stats_held(None) == -1
    # the snapshot mode
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_SCALARS_ONLY) == -5   # profiles need FULL
    assert setgs(nz=0, mask=0) == 0
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_SCALARS_ONLY) == 0
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_NONE) == -5
    assert setgs() == -5                                                     # FULL needed
    assert setgs(ng=0) == 0                                                  # off
    assert L.samsim_b200_set_snapshot_mode(hd, api.SNAP_NONE) == 0
    assert setgs(nz=0, mask=0) == -5
    e.set_snapshot_mode(api.SNAP_FULL)
    e.set_group_stats(goc, DEPTHS[:3], ("T",), max_records=2, ngroup=2)
    # capacity: 2 records; a call that would write a third is refused before anything runs
    e.step(200)
    assert e.group_stats_held() == 2
    clk, launches, th = e.get_clock(), e.launch_count(), e.get_array("thick")
    assert L.samsim_b200_step(hd, 1000) == -5
    assert L.samsim_b200_step(hd, 100) == -5
    assert e.get_clock() == clk and e.launch_count() == launches and pu.same_bits(e.get_array("thick"), th).all()
    e.step(99)   # up to, not onto, the next record
    assert e.group_stats_held() == 2
    # get with ranges, clear
    full = e.group_stats(clear=False)
    one = e.group_stats(clear=False, rec0=1, nrec=1)
    assert list(full["i"]) == [clk["i"] - 100, clk["i"]] and list(one["i"]) == [clk["i"]]
    assert pu.same_bits(one["mean"], full["mean"][1:]).all()
    stats = np.empty(5 * 2 * (NSC + 3))
    assert L.samsim_b200_get_group_stats(hd, api._dp(stats), None, None, 1, 2) == -1
    assert L.samsim_b200_get_group_stats(hd, api._dp(stats), None, None, -1, 1) == -1
    assert L.samsim_b200_get_group_stats(hd, None, None, None, 0, 2) == 0
    assert L.samsim_b200_clear_group_stats(hd) == 0 and e.group_stats_held() == 0
    e.step(1)
    assert e.group_stats_held() == 1
    assert setgs(mx=3) == 0 and e.group_stats_held() == 0   # a new setting drops the held records


def test_large_group_first_record():
    ncol = 67_000
    iout = int(scenarios.sheba_state(200)["i_time_out"])
    e, st = _engine(ncol=ncol, i_time_out=iout, n_time_out=iout)   # the next step writes a record
    goc = np.zeros(ncol, dtype=np.int32)
    goc[np.random.default_rng(5).choice(ncol, 1000, replace=False)] = -1   # 66,000 members
    e.set_group_stats(goc, DEPTHS, ("T", "S_bu"), max_records=1)
    e.step(1)
    s = _snapshot(e, ("thick", "T", "S_bu"))
    h = e.group_stats()
    assert h["count"].shape == (1, 1, NSC + 2 * len(DEPTHS)) and h["count"][0, 0, 0] == 66_000
    ref = reference_record(s, e.status(), np.full(ncol, np.iinfo(np.int64).max), int(h["i"][0]), goc, 1, DEPTHS, ("T", "S_bu"))
    for k, name in enumerate(("count", "mean", "var", "min", "max")):
        assert pu.same_bits(h[name][0], ref[..., k]).all(), name

