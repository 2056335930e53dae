"""The bound pass of gravity drainage on the GPU, bit for bit against the oracle: the columns of
tests/lazy_perm_cases.py in a batch, and one model day of drift of a perturbed ensemble at records 100, 200, 345."""
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
from oracle import parity_util as pu  # noqa: E402
import lazy_perm_cases as lc  # noqa: E402
import scenarios  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("two_pass", [False, True])
@pytest.mark.parametrize("name", sorted(lc.CASES))
def test_bound_pass_cases_on_gpu(oracle_mod, name, two_pass):
    make, chunks, _ = lc.CASES[name]
    col = lc.oracle_column(oracle_mod, make(oracle_mod))
    eng = pu.engine_from_oracle(col, ncol=40)
    eng.set_tuning(two_pass)
    eng.set_forcing(scenarios.sheba_forcing()[None])
    for n in chunks:
        assert col.step(n) == 0
        eng.step(n)
        for c in (0, 39):
            bad = pu.compare_column(col, eng, c, label=f"{name} +{n} col {c}: ")
            assert not bad, "\n".join(bad[:10])
    assert eng.count_failed() == 0


@pytest.mark.parametrize("rec", lc.DRIFT_RECORDS)
def test_bound_pass_one_model_day_of_drift_on_gpu(oracle_mod, rec):
    ncol = 4096
    F = scenarios.sheba_forcing()
    scale, offset, amp = lc.forcing_perturbation(ncol)
    eng = pu.engine_from_oracle(lc.oracle_column(oracle_mod, scenarios.sheba_state(rec)), ncol=ncol)
    eng.set_forcing(F[None], None, scale, offset)
    eng.set_scalar("oflux_amp", amp)
    for n in (1000,) * 8 + (lc.DAY - 8000,):
        eng.step(n)
    assert eng.count_failed() == 0
    for c in np.random.default_rng(rec).choice(ncol, 4, replace=False):
        col = lc.oracle_column(oracle_mod, scenarios.sheba_state(rec), scale[:, c], offset[:, c], amp[c])
        assert col.step(lc.DAY) == 0
        bad = pu.compare_column(col, eng, int(c), label=f"record {rec} col {c}: ")
        assert not bad, "\n".join(bad[:10])
