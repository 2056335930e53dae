"""Cost of per-column forcing series: the bench ensemble (1,048,576 columns, mid-January SHEBA state, the bench's
per-column perturbations) driven by three forcing tables, timed alternately in one process.

  (a) staged    the 9 sites of the bench (<= 16 sites: staged in shared memory per launch)
  (b) global    the same 9 series replicated into 1,048,576 sites, one per column (read in place from global memory)
  (c) distinct  1,048,576 distinct series: site c % 9 started up to 30 days earlier or later, one per column

(b) and (c) would be 96 GB at the full 2,928 records, so every table holds the 64 records around the state's
time_counter and every arm's clock is moved back by the same number of records.  The times are exact integers, so
this changes no result; (a) and (b) read the same values and must stay bitwise identical, which is checked at the end.

    python tools/gpu_many_sites.py [--steps 384] [--reps 4] [--warmup 128]

Prints one JSON line: M column-steps/s per arm (median, min, max over the repetitions), the GPU's name, power limit
and the SM clock sampled during the timed steps.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True
import bench  # noqa: E402  (read-only: state, sites, perturbations, clock sampler)
from samsim_b200 import api  # noqa: E402
from oracle import parity_util as pu  # noqa: E402

NCOL = bench.TOTAL_COLUMNS
NREC_SLICE = 64
MAX_SHIFT = 240   # records: 30 days


def tables(sites: np.ndarray, r0: int):
    """(b) and (c) as [NCOL, 4, NREC_SLICE]: records r0+1 .. r0+NREC_SLICE (1-based) of each column's series"""
    n = sites.shape[2]
    rep = np.empty((NCOL, 4, NREC_SLICE))
    dist = np.empty((NCOL, 4, NREC_SLICE))
    shift = np.random.default_rng(21).integers(-MAX_SHIFT, MAX_SHIFT + 1, NCOL)
    r = np.arange(NREC_SLICE)
    for c0 in range(0, NCOL, 1 << 17):
        c = np.arange(c0, min(c0 + (1 << 17), NCOL))
        rep[c] = sites[:, :, r0:r0 + NREC_SLICE][c % 9]
        idx = (r0 + shift[c, None] + r[None, :]) % n                     # [cols, NREC_SLICE]
        dist[c] = sites[(c % 9)[:, None, None], np.arange(4)[None, :, None], idx[:, None, :]]
    return rep, dist


def engine(st, r0, table, site_of_col):
    cfg = api.Config.from_state(st)
    eng = api.Engine(cfg, NCOL)
    eng.load_column_state(st, 0)
    eng.broadcast_column(0, 0, NCOL)
    eng.set_clock(st["time"] - r0 * 10800.0, st["i"], st["n_time_out"], st["time_counter"] - r0)
    _, scale, offset, amp = bench.perturbations(0, NCOL)
    eng.set_forcing(table, site_of_col, scale, offset)
    eng.set_scalar("oflux_amp", amp)
    return eng


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.strip().split(",")]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=384, help="model steps per timed repetition of each arm")
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=128)
    args = ap.parse_args()
    assert args.reps >= 3 and (args.warmup + args.reps * args.steps) < (NREC_SLICE - 12) * 1080

    st = bench.load_state(bench.START_RECORD)
    sites = bench.load_sites(NREC_SLICE)
    r0 = int(st["time_counter"]) - 9      # the slice starts 8 records before the one read first
    rep, dist = tables(sites, r0)
    site9 = bench.perturbations(0, NCOL)[0]
    own = np.arange(NCOL, dtype=np.int32)
    arms = {"staged": engine(st, r0, sites[:, :, r0:r0 + NREC_SLICE], site9),
            "global": engine(st, r0, rep, own),
            "distinct": engine(st, r0, dist, own)}
    del rep, dist
    for eng in arms.values():
        eng.step(args.warmup)

    times = {k: [] for k in arms}
    sampler = bench.ClockSampler(0)
    sampler.start()
    for _ in range(args.reps):
        for name, eng in arms.items():
            eng.synchronize()
            t0 = time.perf_counter()
            eng.step(args.steps, sync=False)
            eng.synchronize()
            times[name].append(time.perf_counter() - t0)
    sampler.stop_flag.set()
    sampler.join(timeout=2)

    same = []
    a, b = arms["staged"], arms["global"]
    for name in pu.CMP_ARRAYS:
        same.append(bool(pu.same_bits(a.get_array(name), b.get_array(name)).all()))
    for name in api.SCALAR_IDS:
        same.append(bool(pu.same_bits(a.get_scalar(name), b.get_scalar(name)).all()))
    for name in api.INT_IDS:
        same.append(bool(np.array_equal(a.get_int(name), b.get_int(name))))
    failed = {k: e.count_failed() for k, e in arms.items()}

    rate = {}
    for name, ts in times.items():
        r = NCOL * args.steps / np.array(ts) / 1e6
        rate[name] = {"median": float(np.median(r)), "min": float(r.min()), "max": float(r.max()),
                      "spread": float((r.max() - r.min()) / np.median(r)), "all": [round(x, 2) for x in r]}
    line = {"what": "M column-steps/s, 1,048,576 columns, SHEBA state 200 (mid-January), bench perturbations",
            "steps": args.steps, "reps": args.reps, "warmup": args.warmup, "records_per_table": NREC_SLICE,
            "rate": rate, "global_vs_staged": rate["global"]["median"] / rate["staged"]["median"],
            "distinct_vs_staged": rate["distinct"]["median"] / rate["staged"]["median"],
            "staged_equals_global_bitwise": all(same), "failed_columns": failed,
            "gpu": gpu_info(), "clocks": sampler.summary()}
    print(json.dumps(line))
    for name, r in rate.items():
        print(f"{name:9s} {r['median']:7.2f} M column-steps/s  (min {r['min']:.2f}, max {r['max']:.2f})", file=sys.stderr)
    if not all(same):
        raise SystemExit("staged and global tables gave different results")


if __name__ == "__main__":
    main()
