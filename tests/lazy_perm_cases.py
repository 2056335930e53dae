"""Columns for the bound pass of gravity drainage (csrc/physics.cuh, grav_drain_bound): on lean steps the layers above
the topmost layer whose bound can reach ray_crit are not evaluated, so these columns put that layer in every place
that matters.  Shared by tests/test_lazy_perm_cpu.py (device code on the host) and tests/test_lazy_perm_gpu.py.

Each case is (restart record, edit of S_abs, launch chunks).  A launch's last step evaluates every layer exactly
(ray is observable after it); all its other steps take the bound pass."""
from __future__ import annotations

import numpy as np

import scenarios

RAY_CRIT = 4.89  # mo_grav_drain.f90:75


def _scaled(rec: int, j0: int, j1: int, f: float) -> dict:
    st = scenarios.sheba_state(rec)
    a = np.array(st["S_abs"], dtype=np.float64)
    a[j0:j1] *= f
    st["S_abs"] = a
    return st


def oracle_column(oracle_mod, st: dict, scale=None, offset=None, oflux_amp=None):
    F = scenarios.sheba_forcing()
    if scale is not None:
        F = np.stack([F[q] * scale[q] + offset[q] for q in range(4)])
    col = oracle_mod.Column(4, "det")
    col.set_forcing(*F)
    col.load_state(st)
    if oflux_amp is not None:
        col.set_scalar("oflux_amp", oflux_amp)
    return col


def ray_after_one_step(oracle_mod, st: dict) -> np.ndarray:
    col = oracle_column(oracle_mod, st)
    assert col.step(1) == 0
    return col.array("ray")[: col.int("N_active") - 1]


def slack_band_state(oracle_mod) -> dict:
    """Mid-winter column with the salt of layers 41..99 raised until the Rayleigh number of layer 40 -- the layer just
    above the raised ones, 5 blocks above the warm bottom -- lies in [ray_crit (1 - 1e-3), ray_crit (1 - 1e-4)]."""
    lo, hi = 1.0, 1.5
    for _ in range(60):
        f = 0.5 * (lo + hi)
        r = ray_after_one_step(oracle_mod, _scaled(200, 40, 99, f))[39] / RAY_CRIT
        if 1.0 - 1e-3 <= r <= 1.0 - 1e-4:
            return _scaled(200, 40, 99, f)
        lo, hi = (f, hi) if r < 1.0 - 1e-3 else (lo, f)
    raise AssertionError("no factor puts layer 40 into the slack band")


CASES = {
    # name: (state builder, chunks, expected first candidate layer (1-based) after the first step, or None)
    "slack_band": (slack_band_state, (1, 40, 200), None),
    "topmost_candidate_in_block_1": (lambda o: _scaled(200, 0, 99, 3.0), (1, 40, 200), 1),
    "no_candidate": (lambda o: _scaled(200, 0, 99, 0.5), (1, 40, 200), 0),
    "sparse_candidates_melt": (lambda o: scenarios.sheba_state(345), (1, 40, 300), 19),
}

DRIFT_RECORDS = (100, 200, 345)
DAY = 8640  # model steps of 10 s


def forcing_perturbation(ncol: int):
    """the bench's per-column perturbations (bench.py, SURVEY section 8d): scale, offset [4, ncol], oceanic flux amplitude"""
    rng = np.random.default_rng(4)
    scale, offset = np.ones((4, ncol)), np.zeros((4, ncol))
    offset[2] = rng.uniform(-2, 2, ncol)
    scale[1] = rng.uniform(0.95, 1.05, ncol)
    scale[0] = rng.uniform(0.9, 1.1, ncol)
    scale[3] = rng.uniform(0.5, 1.5, ncol)
    return scale, offset, 7.0 * rng.uniform(0.5, 1.5, ncol)
