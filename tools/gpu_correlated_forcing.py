"""Cost of the correlated stochastic forcing (samsim_b200_set_stochastic_forcing_correlated) on the bench ensemble:
1,048,576 columns, mid-January SHEBA state, the bench's per-column perturbations, a record every 360 steps (config 4's
cadence).  The kinds are correlated through CORR in every setting, so every setting runs the two-kernel path.

  kernels      torch.profiler: samsim_noise_basis_kernel and samsim_noise_mix_kernel of step(360) calls (one launch
               each, a window of two records) at nbasis 4,096 and 1,048,576, nmix 1 and 4.  The first call after a new
               setting restarts the window from record 1; the later ones resume from the cursor.
  cold         the restart from record 1 at record 8,000 (a table of 8,100 records, the clock set there), nmix 4 at
               both nbasis: a synchronised step(1) right after a new setting against the step(1) after it, host clock.
  throughput   two identical handles, the feature off and on (nbasis 4,096, nmix 4); step(360) timed with a host clock
               around a synchronised call, the handles alternating and swapping places every repetition.
  registers    `-Xptxas -v` of the two step kernel instances and the noise kernels, compiled here for sm_100a.

    python tools/gpu_correlated_forcing.py [--reps 8] [--out FILE]

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
CORR = np.array([[1.0, -0.6, -0.3, -0.2], [-0.6, 1.0, 0.5, 0.3], [-0.3, 0.5, 1.0, 0.1], [-0.2, 0.3, 0.1, 1.0]])
COLD_REC = 8000
KERNELS = ["samsim_noise_basis_kernel", "samsim_noise_mix_kernel", "samsim_step_kernel"]


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.strip().split(",")]))


def ptxas_report():
    """registers, stack and spills of the step kernel instances and the noise kernels (a compile for sm_100a into a
    temporary directory)"""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as d:
        cmd = [nvcc] + build.NVCC_FLAGS + ["-Xptxas", "-v", "-o", str(Path(d) / "lib.so"), str(build.SRC)]
        r = subprocess.run(cmd, capture_output=True, text=True)
    out, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Function properties for (_Z\d+(samsim_step_kernel|samsim_noise_\w+?kernel)\w*)", line)
        if m:
            cur = m.group(1)
            continue
        if cur and "spill stores" in line:
            s = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
            out[cur] = {"stack": int(s.group(1)), "spill_stores": int(s.group(2)), "spill_loads": int(s.group(3))}
        elif cur and "Used" in line:
            out[cur]["registers"] = int(re.search(r"Used (\d+) registers", line).group(1))
            cur = None
    return out or {"error": r.stderr[-2000:]}


def mixing(nbasis, nmix):
    """column c mixes ids (c + m * nbasis / nmix) % nbasis, m < nmix: distinct, every id used; normal weights scaled to
    unit norm, so every column's noise has the variance sigma^2 of the single-stream setting"""
    c = np.arange(NCOL, dtype=np.int64)
    basis = np.stack([(c + m * (nbasis // nmix)) % nbasis for m in range(nmix)], axis=1).astype(np.int32)
    w = np.random.default_rng(nbasis + nmix).normal(size=basis.shape)
    return basis, w / np.sqrt((w * w).sum(axis=1, keepdims=True))


def set_noise(eng, nbasis, nmix):
    basis, w = mixing(nbasis, nmix)
    eng.set_stochastic_forcing(SEED, SIGMA, PHI, MODE, corr=CORR, basis=basis, weights=w)


def make_engine(st, sites, noise):
    eng = bench.make_engine(api, {**st, "i_time_out": IOUT, "n_time_out": IOUT}, sites, NCOL, 0, 0)
    eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)
    if noise:
        set_noise(eng, 4096, 4)
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
    ap.add_argument("--reps", type=int, default=8, help="timed step(360) calls per arm")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    st = bench.load_state(bench.START_RECORD)
    sites = bench.load_sites(64)
    off, on = make_engine(st, sites, False), make_engine(st, sites, True)
    for eng in (off, on):
        eng.step(IOUT + 1)   # warm up
    res = {"what": "correlated stochastic forcing on 1,048,576 columns, SHEBA state 200 (mid-January), bench "
                   "perturbations, a record every 360 steps; sigma %s, phi %s, mode %s, corr %s"
                   % (SIGMA, PHI, MODE, CORR.tolist())}

    times = {"off": [], "on": []}
    for rep in range(args.reps):
        for arm, eng in ((("off", off), ("on", on)) if rep % 2 == 0 else (("on", on), ("off", off))):
            eng.synchronize()
            t0 = time.perf_counter()
            eng.step(IOUT + 1, sync=False)
            eng.synchronize()
            times[arm].append(time.perf_counter() - t0)
    a, b = np.array(times["on"]), np.array(times["off"])
    res["throughput_360"] = {"nbasis": 4096, "nmix": 4, "s_on": a.tolist(), "s_off": b.tolist(),
                             "Mcolsteps_off": NCOL * (IOUT + 1) / np.median(b) / 1e6,
                             "Mcolsteps_on": NCOL * (IOUT + 1) / np.median(a) / 1e6,
                             "cost": float(np.median(a) / np.median(b) - 1.0),
                             "spread_off": float(np.ptp(b) / np.median(b)), "spread_on": float(np.ptp(a) / np.median(a))}
    print(json.dumps(res["throughput_360"]), file=sys.stderr)

    res["kernels_360"] = []
    for nbasis in (4096, NCOL):
        for nmix in (1, 4):
            set_noise(on, nbasis, nmix)
            k = kernel_ms(lambda: [on.step(IOUT + 1, sync=False) for _ in range(3)], KERNELS)
            row = {"nbasis": nbasis, "nmix": nmix, "basis_ms": k[KERNELS[0]], "mix_ms": k[KERNELS[1]],
                   "step_ms": k[KERNELS[2]], "first_call": "restarts from record 1"}
            res["kernels_360"].append(row)
            print(json.dumps(row), file=sys.stderr)

    # cold restart at record ~8,000: a table of 8,100 records, the clock just past the start of record COLD_REC - 1
    site, scale, offset, _ = bench.perturbations(0, NCOL)
    reps = -(-8100 // sites.shape[2])
    long = np.concatenate([sites] * reps, axis=2)[:, :, :8100]
    off.set_forcing(long, site, scale, offset)
    clk = off.get_clock()
    off.set_clock((COLD_REC - 2) * 10800.0 + 10.0, clk["i"], clk["n_time_out"], COLD_REC - 1)
    res["cold_restart"] = []

    def step1():
        off.synchronize()
        t0 = time.perf_counter()
        off.step(1)
        return (time.perf_counter() - t0) * 1e3

    for nbasis in (4096, NCOL):
        set_noise(off, nbasis, 4)
        step1()   # module load, first launch
        row = {"record": COLD_REC, "nbasis": nbasis, "nmix": 4, "normals": 4 * nbasis * COLD_REC,
               "ms_restart": [], "ms_next": []}
        for _ in range(3):
            set_noise(off, nbasis, 4)   # a new setting: the next window restarts from record 1
            row["ms_restart"].append(step1())
            row["ms_next"].append(step1())
        res["cold_restart"].append(row)
        print(json.dumps(row), file=sys.stderr)

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
