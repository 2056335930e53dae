"""bench.py --dump-outputs: the files hold what the timed path computed in its last step, the same bits on every run
with the same arguments, and the step count they reflect is the one --steps and --warmup ask for."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent

pytestmark = pytest.mark.gpu

NCOL, STEPS, WARMUP = 2048, 2, 3


def _bench(out_dir):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--columns", str(NCOL), "--steps", str(STEPS),
                        "--warmup", str(WARMUP), "--no-year-weighted", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == STEPS
    return {p.stem: np.load(p) for p in sorted(out_dir.glob("*.npy"))}


def test_dump_outputs_repeat_and_match_the_engine(tmp_path):
    sys.path.insert(0, str(ROOT))
    import bench
    from samsim_b200 import api
    a, b = _bench(tmp_path / "a"), _bench(tmp_path / "b")
    assert a.keys() == b.keys()
    assert {"thickness", "T_top", "N_active", "status", "ensemble_reduction", "profile_columns", "profile_T"} <= a.keys()
    for name, x in a.items():
        assert x.dtype in (np.float32, np.float64), name
        assert np.array_equal(x, b[name], equal_nan=True), name
    assert sum(x.nbytes for x in a.values()) <= bench.DUMP_MAX_BYTES
    # the same columns advanced by warmup + 2 x steps bench steps (device-resident and end-to-end regions)
    eng = bench.make_engine(api, bench.load_state(bench.START_RECORD), bench.load_sites(64), NCOL, 0, 0)
    for _ in range(WARMUP + 2 * STEPS):
        eng.step(bench.MODEL_STEPS)
    for name in ("thickness", "bulk_salin", "freeboard", "thick_snow", "T_top"):
        assert np.array_equal(a[name], eng.get_scalar(name)), name
    assert np.array_equal(a["N_active"], eng.get_int("N_active").astype(np.float32))
    cols = a["profile_columns"].astype(np.int64)
    assert len(cols) == bench.DUMP_PROFILE_COLUMNS and np.array_equal(cols, bench.column_sample(NCOL, bench.DUMP_PROFILE_COLUMNS, 1))
    for name in bench.DUMP_PROFILES:
        assert np.array_equal(a[f"profile_{name}"], eng.get_array(name)[cols]), name
    eng.close()
