"""The bound pass of gravity drainage on the device code compiled for the host, bit for bit against the oracle:
a layer just below ray_crit above the drained region, the topmost candidate in block 1, no candidate at all, the
sparse candidates of the melt season, and one model day of drift under per-column forcing (tests/lazy_perm_cases.py)."""
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
from hostbuild import hostkernel as hk  # noqa: E402
from oracle import parity_util as pu  # noqa: E402
import lazy_perm_cases as lc  # noqa: E402
import scenarios  # noqa: E402


def _host(col, F, two_pass, scale=None, offset=None):
    k = hk.HostKernel(pu.config_from_oracle(col))
    k.load_state(col.state())
    k.set_tuning(two_pass)
    if scale is None:
        k.set_forcing(F)
    else:
        k.set_forcing(F, scale, offset)
    return k


@pytest.mark.parametrize("two_pass", [False, True])
@pytest.mark.parametrize("name", sorted(lc.CASES))
def test_bound_pass_cases_on_host(oracle_mod, name, two_pass):
    make, chunks, first = lc.CASES[name]
    st = make(oracle_mod)
    if first is not None:
        r = lc.ray_after_one_step(oracle_mod, st)
        got = int(np.argmax(r > lc.RAY_CRIT)) + 1 if (r > lc.RAY_CRIT).any() else 0
        assert got == first, (name, got)
    col = lc.oracle_column(oracle_mod, st)
    k = _host(col, scenarios.sheba_forcing(), two_pass)
    for n in chunks:
        assert col.step(n) == 0 and k.step(n) == 0
        bad = pu.compare_column(col, k, 0, label=f"{name} +{n}: ")
        assert not bad, "\n".join(bad[:10])


@pytest.mark.parametrize("rec", lc.DRIFT_RECORDS)
def test_bound_pass_one_model_day_of_drift_on_host(oracle_mod, rec):
    """one day (8,640 steps, launches of 1,000) of sampled columns of the bench ensemble"""
    F = scenarios.sheba_forcing()
    scale, offset, amp = lc.forcing_perturbation(64)
    for c in (5, 41):
        col = lc.oracle_column(oracle_mod, scenarios.sheba_state(rec), scale[:, c], offset[:, c], amp[c])
        k = _host(col, F, False, scale[:, c], offset[:, c])
        k.set_scalar("oflux_amp", amp[c])
        for n in (1000,) * 8 + (lc.DAY - 8000,):
            assert col.step(n) == 0 and k.step(n) == 0
        bad = pu.compare_column(col, k, 0, label=f"record {rec} col {c}: ")
        assert not bad, "\n".join(bad[:10])
