"""Cost of the per-column time statistics (samsim_b200_set_time_stats) on the bench ensemble: 1,048,576 columns,
mid-January SHEBA state, the bench's per-column perturbations, a record every 360 steps (config 4's cadence), Q = 20
(the snapshot scalars) and Q = 120 (plus T and S_bu on 50 depths).

  kernel       torch.profiler: the time of every samsim_ts_record_kernel launch over windows of three records, by its
               place in the window (opening: accumulators written only; middle: read and written; closing: read, and
               the finalised window written into the history), and of samsim_ts_close_kernel; unbinned and re-binned.
               Every step is made an output step (set_clock) and step(1) is called once per record.
  per record   two identical handles, statistics on and off; step(1) on an output step timed with the handles' CUDA
               events (last_step_ms), alternating; the difference is the statistics' time per record.
  bytes        what the record kernel must move per record, counted in `bytes_per_record` from the snapshot's N_active
               and ice thickness, over the kernel time: the share of the 7.7 TB/s of HBM3e.
  throughput   step(360) with one record at its last step, the two handles alternating in one process, windows of
               24 records (one model day).

    python tools/gpu_time_stats.py [--records 24] [--reps 3] [--out FILE]

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
NSC = len(api.SNAP_SCALARS)
SETS = {"Q20": ((), ()), "Q120": (DEPTHS, ("T", "S_bu"))}   # depths, profiles
HBM_BYTES_PER_S = 7.7e12
KINDS = ("opening", "middle", "closing")


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.strip().split(",")]))


def bytes_per_record(eng, depths, profiles, binned):
    """DRAM bytes samsim_ts_record_kernel needs for one record, every column contributing, by the record's place:
    all      status (4), slot_of_col when re-binned (4), the 20 scalars (8 each); with profiles N_active, thick of layers
             1..N_active and one value per profile and depth above the ice bottom (8 each)
    opening  writes n, mean, M2, min, max of every quantity (5 x 8)
    middle   reads and writes them for the quantities the column reaches (2 x 5 x 8)
    closing  reads them and writes the finalised window into the history, for every quantity (2 x 5 x 8)"""
    s = eng.get_snapshot(arrays=False)
    na = s["N_active"].astype(np.float64)
    reached = np.searchsorted(depths, s["thickness"], side="right").astype(np.float64) if len(profiles) else np.zeros(NCOL)
    Q = NSC + len(profiles) * len(depths)
    common = NCOL * (4 + (4 if binned else 0) + 8 * NSC)
    if profiles:
        common += 8 * (NCOL + na.sum() + len(profiles) * reached.sum())
    reached_q = NSC * NCOL + len(profiles) * reached.sum()
    return {"opening": float(common + 40 * Q * NCOL), "middle": float(common + 80 * reached_q),
            "closing": float(common + 80 * Q * NCOL)}


def make_engine(st, sites):
    eng = bench.make_engine(api, {**st, "i_time_out": IOUT, "n_time_out": IOUT}, sites, NCOL, 0, 0)
    eng.set_snapshot_mode(api.SNAP_FULL)
    return eng


def one_record(eng):
    clk = eng.get_clock()
    eng.set_clock(clk["time"], clk["i"], IOUT, clk["time_counter"])   # the next step writes a record
    eng.step(1)


def per_record(on, off, records):
    """step(1) on an output step of two identical handles, statistics on / off, alternating: ms per record by the
    record's place in its window of three"""
    t = {"off": []} | {k: [] for k in KINDS}
    on.clear_time_stats()
    for r in range(3 * records + 3):
        for arm, eng in (("on", on), ("off", off)):
            if arm == "on" and on.time_stats_held() >= 2:
                on.clear_time_stats()
            one_record(eng)
            if r >= 3:   # the first window warms up
                t[KINDS[r % 3] if arm == "on" else "off"].append(eng.last_step_ms())
    off_ms = float(np.median(t["off"]))
    out = {"ms_off": off_ms, "ms_off_spread": float(np.ptp(t["off"]))}
    for k in KINDS:
        out[f"ms_on_{k}"] = float(np.median(t[k]))
        out[f"ms_stats_{k}"] = float(np.median(t[k]) - off_ms)
    return out


def kernel_times(eng, records):
    """device time of each statistics kernel launch from torch.profiler (CUPTI), ms, by the record's place in its
    window of three; then one samsim_b200_close_time_window after a middle record"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    eng.clear_time_stats()
    one_record(eng)
    one_record(eng)
    one_record(eng)   # a window of three is complete: the next record opens one
    eng.clear_time_stats()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for r in range(3 * records):
            if eng.time_stats_held() >= 2:
                eng.clear_time_stats()
            one_record(eng)
        eng.clear_time_stats()
        one_record(eng)
        one_record(eng)
        eng.close_time_window()
        eng.synchronize()
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if "samsim_ts_" in e.name), key=lambda e: e.time_range.start)
    rec = [e.time_range.elapsed_us() / 1e3 for e in ev if "samsim_ts_record_kernel" in e.name]
    close = [e.time_range.elapsed_us() / 1e3 for e in ev if "samsim_ts_close_kernel" in e.name]
    out = {"launches_record": len(rec), "launches_close": len(close)}
    if len(rec) == 3 * records + 2:
        for j, k in enumerate(KINDS):
            out[f"ms_{k}"] = float(np.median(rec[j:3 * records:3]))
    else:   # the profiler's event list is not one per launch: report the totals only
        out["ms_record_mean"] = float(np.mean(rec)) if rec else None
    out["ms_close_window"] = close[-1] if close else None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=24, help="timed windows of three records per setting and arm")
    ap.add_argument("--reps", type=int, default=3, help="360-step calls per arm in the throughput comparison")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    st = bench.load_state(bench.START_RECORD)
    sites = bench.load_sites(64)
    on, off = make_engine(st, sites), make_engine(st, sites)   # identical handles: statistics on / off
    for eng in (on, off):
        eng.step(IOUT + 1)   # warm up: one record
    res = {"what": "per-column time statistics on 1,048,576 columns, SHEBA state 200 (mid-January), bench "
                   "perturbations; Q = 20 (the snapshot scalars) and Q = 120 (+ T, S_bu on 50 depths)",
           "records": args.records, "settings": {}}
    for binned in (False, True):
        if binned:
            on.set_time_stats(0, [])
            for eng in (on, off):
                eng.step(2 * (IOUT + 1))   # let the columns drift apart, then sort them
                res["rebin_changed_order"] = eng.rebin()
        for name, (depths, profiles) in SETS.items():
            on.set_time_stats(3, None, depths, profiles, max_windows=2)
            r = per_record(on, off, args.records)
            r["kernels"] = kernel_times(on, max(4, args.records // 2))
            b = bytes_per_record(on, np.asarray(depths), profiles, binned)
            r["bytes"] = b
            for k in KINDS:
                ms = r["kernels"].get(f"ms_{k}")
                r[f"hbm_share_{k}"] = b[k] / (ms * 1e-3) / HBM_BYTES_PER_S if ms else None
            res["settings"][name + (" rebinned" if binned else "")] = r
            print(name, "rebinned" if binned else "unbinned", json.dumps(r), file=sys.stderr)

    # throughput at the 360-step cadence: one record per call, daily windows, the two handles alternating
    thr = {}
    for name, (depths, profiles) in SETS.items():
        on.set_time_stats(24, None, depths, profiles, max_windows=1)
        times = {"on": [], "off": []}
        for _ in range(args.reps + 1):
            for arm, eng in (("off", off), ("on", on)):
                clk = eng.get_clock()
                eng.set_clock(clk["time"], clk["i"], 0, clk["time_counter"])   # a record at the call's last step
                eng.synchronize()
                t0 = time.perf_counter()
                eng.step(IOUT + 1, sync=False)
                eng.synchronize()
                times[arm].append(time.perf_counter() - t0)
        a, b = np.array(times["on"][1:]), np.array(times["off"][1:])
        thr[name] = {"s_on": a.tolist(), "s_off": b.tolist(),
                     "Mcolsteps_off": NCOL * (IOUT + 1) / np.median(b) / 1e6,
                     "Mcolsteps_on": NCOL * (IOUT + 1) / np.median(a) / 1e6,
                     "cost": float(np.median(a) / np.median(b) - 1.0)}
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
