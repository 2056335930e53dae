"""Cost of the group statistics (samsim_b200_set_group_stats) on the bench ensemble: 1,048,576 columns, mid-January
SHEBA state, the bench's per-column perturbations, a record every 360 steps (config 4's cadence), the 20 snapshot
scalars plus T and S_bu on 50 depths (Q = 120).

  per record   two identical handles, statistics on and off; every step is made an output step (set_clock) and
               step(1) is timed with the handles' CUDA events (last_step_ms), alternating; the difference is the
               statistics kernels' time per record.  torch.profiler, in a separate pass, gives the time of each statistics kernel.
               Group layouts 1 x 1,048,576, 1,024 x 1,024, 65,536 x 16 and 1,048,576 x 1, unbinned and re-binned.
  throughput   step(360) with one record at its last step, the two handles alternating in one process.
  bytes        what the kernels must move per record, counted from the snapshot (N_active, ice thickness) by the
               model in `bytes_per_record`, over the kernel time: the share of the 7.7 TB/s of HBM3e.

    python tools/gpu_group_stats.py [--records 24] [--reps 3] [--out FILE]

Prints one JSON line (also written to --out) with the GPU's name and power limit read in the same run.
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
import bench  # noqa: E402  (read-only: state, sites, perturbations)
from samsim_b200 import api  # noqa: E402

NCOL = bench.TOTAL_COLUMNS
IOUT = 359
DEPTHS = np.linspace(0.04, 2.0, 50)
PROFILES = ("T", "S_bu")
Q = len(api.SNAP_SCALARS) + len(PROFILES) * len(DEPTHS)
HBM_BYTES_PER_S = 7.7e12
LAYOUTS = {"1x1048576": 1, "1024x1024": 1024, "65536x16": 65536, "1048576x1": NCOL}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.strip().split(",")]))


def bytes_per_record(eng, ngroup):
    """DRAM bytes the five statistics kernels need for one record (every member contributing):
    gather    reads col, status (4 + 4), the 20 snapshot scalars, thick of layers 1..N_active, one value per profile
              and reached depth; writes the reached quantities and reach (8 each)
    tile x 2  read info (4), reach (8) and the Q values (8 each); pass 2 also reads the group means (8 per group and q)
    results   count, mean, min, max, then variance: 5 doubles per group and quantity (written once, mean read once)"""
    s = eng.get_snapshot(arrays=False)
    na = s["N_active"].astype(np.float64)
    reached = np.searchsorted(DEPTHS, s["thickness"], side="right").astype(np.float64)   # depths above the ice bottom
    npad = NCOL   # every layout here is a power of two: no padding
    gather = npad * (4 + 4 + 8) + 8 * (20 * NCOL + na.sum() + len(PROFILES) * reached.sum()) + \
        8 * (20 * NCOL + len(PROFILES) * reached.sum())
    tiles = 2 * npad * (4 + 8 + 8 * Q) + 8 * ngroup * Q
    results = 8 * ngroup * Q * (5 + 1)
    return float(gather + tiles + results)


def make_engine(st, sites):
    eng = bench.make_engine(api, {**st, "i_time_out": IOUT, "n_time_out": IOUT}, sites, NCOL, 0, 0)
    eng.set_snapshot_mode(api.SNAP_FULL)
    return eng


def groups(ngroup):
    return (np.arange(NCOL) // (NCOL // ngroup)).astype(np.int32)


def per_record(on, off, records):
    """step(1) on an output step of two identical handles, statistics on / off, alternating: ms per record"""
    t = {"on": [], "off": []}
    for _ in range(records + 1):
        for arm, eng in (("on", on), ("off", off)):
            clk = eng.get_clock()
            eng.set_clock(clk["time"], clk["i"], IOUT, clk["time_counter"])   # the next step writes a record
            eng.clear_group_stats()
            eng.step(1)
            t[arm].append(eng.last_step_ms())
    a, b = np.array(t["on"][1:]), np.array(t["off"][1:])   # the first of each arm warms up
    return {"ms_on": float(np.median(a)), "ms_off": float(np.median(b)), "ms_stats": float(np.median(a) - np.median(b)),
            "ms_on_spread": float(a.max() - a.min()), "ms_off_spread": float(b.max() - b.min())}


def kernel_times(eng, records):
    """per-kernel device time of the statistics kernels from torch.profiler (CUPTI), ms per record"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(records):
            clk = eng.get_clock()
            eng.set_clock(clk["time"], clk["i"], IOUT, clk["time_counter"])
            eng.clear_group_stats()
            eng.step(1)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "samsim_gs_" in ev.key:
            name = ev.key.split("(")[0].replace("void ", "")
            out[name] = out.get(name, 0.0) + ev.device_time_total / 1e3 / records
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=24, help="timed records per layout and arm")
    ap.add_argument("--reps", type=int, default=3, help="360-step calls per arm in the throughput comparison")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    st = bench.load_state(bench.START_RECORD)
    sites = bench.load_sites(64)
    on, off = make_engine(st, sites), make_engine(st, sites)   # identical handles: statistics on / off
    for eng in (on, off):
        eng.step(IOUT + 1)   # warm up: one record
    res = {"what": "group statistics on 1,048,576 columns, SHEBA state 200 (mid-January), bench perturbations, "
                   f"Q = {Q} (20 scalars + T, S_bu on 50 depths)", "records": args.records, "layouts": {}}
    for binned in (False, True):
        if binned:
            on.set_group_stats(ngroup=0)
            for eng in (on, off):
                eng.step(2 * (IOUT + 1))   # let the members drift apart, then sort them
                res["rebin_changed_order"] = eng.rebin()
        for name, ngroup in LAYOUTS.items():
            on.set_group_stats(groups(ngroup), DEPTHS, PROFILES, max_records=1)
            r = per_record(on, off, args.records)
            r["kernels_ms"] = kernel_times(on, max(4, args.records // 3))
            kt = sum(r["kernels_ms"].values())
            b = bytes_per_record(on, ngroup)
            r.update(bytes=b, kernel_ms_total=kt, hbm_share=b / (kt * 1e-3) / HBM_BYTES_PER_S if kt > 0 else None)
            res["layouts"][name + (" rebinned" if binned else "")] = r
            print(name, "rebinned" if binned else "unbinned", json.dumps(r), file=sys.stderr)

    # throughput at the 360-step cadence: one record per call, the two handles alternating
    thr = {}
    for name in ("1024x1024", "1048576x1"):
        on.set_group_stats(groups(LAYOUTS[name]), DEPTHS, PROFILES, max_records=1)
        times = {"on": [], "off": []}
        for _ in range(args.reps + 1):
            for arm, eng in (("off", off), ("on", on)):
                clk = eng.get_clock()
                eng.set_clock(clk["time"], clk["i"], 0, clk["time_counter"])   # a record at the call's last step
                eng.clear_group_stats()
                eng.synchronize()
                t0 = time.perf_counter()
                eng.step(IOUT + 1, sync=False)
                eng.synchronize()
                times[arm].append(time.perf_counter() - t0)
        a, b = np.array(times["on"][1:]), np.array(times["off"][1:])
        thr[name] = {"s_on": a.tolist(), "s_off": b.tolist(),
                     "Mcolsteps_off": NCOL * (IOUT + 1) / np.median(b) / 1e6,
                     "Mcolsteps_on": NCOL * (IOUT + 1) / np.median(a) / 1e6,
                     "cost": float(np.median(a) / np.median(b) - 1.0), "records_on": on.group_stats_held()}
        print(name, json.dumps(thr[name]), file=sys.stderr)
    res["throughput_360"] = thr
    res["failed_columns"] = {"on": on.count_failed(), "off": off.count_failed()}
    res["gpu"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
