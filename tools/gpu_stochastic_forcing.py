"""Cost of the stochastic forcing perturbations (samsim_b200_set_stochastic_forcing) on the bench ensemble: 1,048,576
columns, mid-January SHEBA state, the bench's per-column perturbations, a record every 360 steps (config 4's cadence).

  throughput   two identical handles, the feature off and on (multiplicative SW, additive LW and T2m, lognormal
               precip); step(360) timed with a host clock around a synchronised call, the handles alternating.
  kernels      torch.profiler: samsim_noise_kernel and samsim_step_kernel of step(360) calls of the handle with the
               feature on (one launch each, a window of two records).
  cold         the window restarting from record 1 at record ~8,000 (a table of 8,100 records, the clock set there):
               samsim_noise_kernel of the first launch, against the next one that resumes from the cursor.
  registers    `-Xptxas -v` of the two step kernel instances, compiled here for sm_100a.

    python tools/gpu_stochastic_forcing.py [--reps 4] [--out FILE]

Prints one JSON line (also written to --out) with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True
import bench  # noqa: E402  (read-only: state, sites, perturbations)
from samsim_b200 import api, build  # noqa: E402

NCOL = bench.TOTAL_COLUMNS
IOUT = 359
SEED = 20261022
SIGMA, PHI, MODE = [0.25, 12.0, 1.5, 0.6], [0.7, 0.8, 0.9, 0.5], [1, 0, 0, 2]
COLD_REC = 8000


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.strip().split(",")]))


def ptxas_report():
    """registers, stack and spills of the two step kernel instances (a compile for sm_100a into a temporary directory)"""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as d:
        cmd = [nvcc] + build.NVCC_FLAGS + ["-Xptxas", "-v", "-o", str(Path(d) / "lib.so"), str(build.SRC)]
        r = subprocess.run(cmd, capture_output=True, text=True)
    out, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Function properties for (_Z18samsim_step_kernelILb([01])EEv7KParams)", line)
        if m:
            cur = "two_pass" if m.group(2) == "1" else "general"
            continue
        if cur and "spill stores" in line:
            s = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
            out[cur] = {"stack": int(s.group(1)), "spill_stores": int(s.group(2)), "spill_loads": int(s.group(3))}
        elif cur and "Used" in line:
            out[cur]["registers"] = int(re.search(r"Used (\d+) registers", line).group(1))
            cur = None
    return out or {"error": r.stderr[-2000:]}


def make_engine(st, sites, noise):
    eng = bench.make_engine(api, {**st, "i_time_out": IOUT, "n_time_out": IOUT}, sites, NCOL, 0, 0)
    eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    if noise:
        eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE)
    return eng


def kernel_ms(fn, names):
    """device time of each launch of the named kernels while fn() runs (torch.profiler), ms"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {n: [e.time_range.elapsed_us() / 1e3 for e in sorted(prof.events(), key=lambda e: e.time_range.start) if n in e.name]
            for n in names}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=4, help="timed step(360) calls per arm")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    st = bench.load_state(bench.START_RECORD)
    sites = bench.load_sites(64)
    off, on = make_engine(st, sites, False), make_engine(st, sites, True)
    for eng in (off, on):
        eng.step(IOUT + 1)   # warm up
    res = {"what": "stochastic forcing on 1,048,576 columns, SHEBA state 200 (mid-January), bench perturbations, "
                   "a record every 360 steps; sigma %s, phi %s, mode %s" % (SIGMA, PHI, MODE)}

    times = {"off": [], "on": []}
    for _ in range(args.reps):
        for arm, eng in (("off", off), ("on", on)):
            eng.synchronize()
            t0 = time.perf_counter()
            eng.step(IOUT + 1, sync=False)
            eng.synchronize()
            times[arm].append(time.perf_counter() - t0)
    a, b = np.array(times["on"]), np.array(times["off"])
    res["throughput_360"] = {"s_on": a.tolist(), "s_off": b.tolist(),
                             "Mcolsteps_off": NCOL * (IOUT + 1) / np.median(b) / 1e6,
                             "Mcolsteps_on": NCOL * (IOUT + 1) / np.median(a) / 1e6,
                             "cost": float(np.median(a) / np.median(b) - 1.0),
                             "spread_off": float(np.ptp(b) / np.median(b)), "spread_on": float(np.ptp(a) / np.median(a))}
    print(json.dumps(res["throughput_360"]), file=sys.stderr)

    k = kernel_ms(lambda: [on.step(IOUT + 1, sync=False) for _ in range(2)], ["samsim_noise_kernel", "samsim_step_kernel"])
    res["kernels_360"] = {"noise_ms": k["samsim_noise_kernel"], "step_ms": k["samsim_step_kernel"]}
    print(json.dumps(res["kernels_360"]), file=sys.stderr)

    # cold restart at record ~8,000: a table of 8,100 records, the clock just past the start of record COLD_REC - 1
    site, scale, offset, _ = bench.perturbations(0, NCOL)
    reps = -(-8100 // sites.shape[2])
    long = np.concatenate([sites] * reps, axis=2)[:, :, :8100]
    off.set_forcing(long, site, scale, offset)
    off.set_stochastic_forcing(SEED, SIGMA, PHI, MODE)
    clk = off.get_clock()
    off.set_clock((COLD_REC - 2) * 10800.0 + 10.0, clk["i"], clk["n_time_out"], COLD_REC - 1)
    off.step(1)   # the window's cold start, outside the profiler (module load, first launch)
    off.set_stochastic_forcing(SEED, SIGMA, PHI, MODE)   # a new setting: the next window restarts from record 1
    k = kernel_ms(lambda: [off.step(1, sync=False) for _ in range(2)], ["samsim_noise_kernel"])["samsim_noise_kernel"]
    res["cold_restart"] = {"record": COLD_REC, "normals": 4 * NCOL * COLD_REC, "noise_ms_restart": k[0] if k else None,
                           "noise_ms_next": k[1] if len(k) > 1 else None}
    print(json.dumps(res["cold_restart"]), file=sys.stderr)

    res["failed_columns"] = {"on": on.count_failed(), "off": off.count_failed()}
    res["registers"] = ptxas_report()
    res["gpu"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
