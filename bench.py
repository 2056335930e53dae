#!/usr/bin/env python
"""bench.py -- column-timesteps/sec of the SAMSIM column timestep on 1..8 B200.

Workload (BASELINE.json config 5): 1,048,576 ERA-interim-style columns (testcase-4 flags, 100 layers, dt 10 s) PER
GPU: the columns are independent, so the ensemble is sharded over the N ranks with no data-path collective and the
bench reports weak scaling (N x 1,048,576 columns on N GPUs; `--scaling strong` shards a fixed total instead, which
at 8 GPUs leaves 131,072 columns = 0.86 of a wave per GPU).  Every column starts from the oracle's SHEBA state
of mid January (output record 200: N_active = 100, 0.124 m of snow) and gets its own forcing: base site c mod 9 of
input/ERA-interim, T2m + U(-2,2) K, fl_lw x U(.95,1.05), fl_sw x U(.9,1.1), precip x U(.5,1.5), oceanic flux
amplitude 7 x U(.5,1.5) W/m2 (default_rng(4), SURVEY section 8d).

One bench "step" = MODEL_STEPS consecutive model timesteps of every column of the rank (one kernel launch).
  value  : column-timesteps/s with the state resident in HBM, CUDA events on the launching stream, max over ranks
  e2e    : the same through the C ABI with HOST buffers inside the timed region: every step uploads the forcing
           table (pinned host memory -> samsim_b200_update_forcing), runs samsim_b200_step, and reads back five
           per-column diagnostics (pinned host memory) plus the 18-number ensemble reduction.
  roofline: FP64 vector pipe.  achieved = F_ALG x column-steps/s; peak = DFMA micro-benchmark run live on the same
           GPU (MEASURED_PEAKS.json has no FP64 entry); HBM view alongside (peak from MEASURED_PEAKS.json).
  roofline.issue_ceiling: the FP64 pipe issues one instruction per lane and clock whether it is a DADD, a DMUL or a
           DFMA, and the bit-exact contract (-fmad=false) forbids contracting a*b+c: the DFMA peak (2 flop per slot)
           is not reachable by construction.  issue_ceiling = 148 SMs x 64 lanes x SM clock / (FP64 instructions per
           column-step from the committed ncu capture) is the throughput at which the FP64 pipe would be saturated;
           roofline.hw_tflops is what the hardware executed (dadd + dmul + 2 dfma), next to the algorithmic rate.
  strong : (N > 1) the same 1,048,576-column ensemble sharded over the N ranks (fixed total), timed the same way.
  year_weighted: (N = 1) throughput over the regimes of a SHEBA year instead of the mid-winter state alone: six
           ensembles start from the oracle states of records 60 / 100 / 200 / 330 / 345 / 400, drift 8,640 steps (one
           model day) under per-column forcing with divergence-driven re-binning, are timed for 640 more steps, and are combined
           with the share of the golden run's 1,643 records that each regime represents (harmonic mean = time-weighted).
  cpu_baseline / --impl reference: the CPU oracle (C port of the Fortran; no Fortran compiler exists in this image),
           one column per OS thread on all host cores, on a bounded sample of the same columns; the libm build (what
           the reference binary links) is the one that is timed, the deterministic-math build is reported beside it.

--dump-outputs DIR (rank 0): after the timed steps, what the end-to-end path handed its caller in its last step --
the five per-column diagnostics and the 18-number ensemble reduction -- plus N_active and status of every column and
the layer profiles of a seeded sample of columns, as DIR/<name>.npy (float64; N_active and status float32), about
55 MB at the default size.  Beyond 1,048,576 columns the per-column files hold a seeded sample, listed in
columns.npy.  The inputs are seeded, so two builds run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True   # the bench writes nothing into the tree, which may be read-only

TOTAL_COLUMNS = 1 << 20
MODEL_STEPS = 64            # model timesteps per bench step (one launch)
START_RECORD = 200          # oracle SHEBA state (tests/golden/sheba_oracle_states.npz)
SITES = ["sheba", "70N00W", "75N00W", "75N180E", "80N00E", "80N90E", "85N180E", "NorthPole", "barrow"]
# Algorithmic FP64 work of ONE column timestep of this workload, counted on the CPU oracle with the
# operation-counting build (python tools/count_flops.py; DESIGN.md section 5): the reference algorithm as written
# executes 50775 add/sub + 49926 mul + 12229 div = 112930 flop (+ 103 pow, 201 exp, 1 sin calls, not counted)
# per column-timestep from the mid-January SHEBA state (N_active = 100).
F_ALG_FLOP_PER_COLUMN_STEP = 112930.0
B_ALG_BYTES_PER_COLUMN_STEP = 2 * 4 * 100 * 8  # read+write of m, S_abs, H_abs, thick once per model step
NCU_DIGEST = "r2_ncu_step_kernel.json"           # committed ncu --set full digest of samsim_step_kernel
NCU_DIGEST_COLUMN_STEPS = 262144 * 64            # columns x model steps of the launch captured there
# Regimes of the SHEBA year: oracle restart record -> share of the golden run's 1,643 records it represents
# (reference_output/Reference_SHEBA_with_Version_2: N_active from dat_thick, melt from dat_melt; classification in
# DESIGN.md section 6: open water N_active = 1; ice melt with / without a full grid; snow melt; growth; full-grid winter)
YEAR_REGIMES = [(200, "winter, grid full", 0.6190), (345, "bare-ice melt, flushing", 0.1382), (100, "growth, grid filling", 0.1181),
                (400, "late-summer melt, grid shrinking", 0.0493), (60, "open water / freeze-up", 0.0402),
                (330, "melt onset, wet snow", 0.0353)]
YEAR_COLUMNS = 151552            # one full wave of the step kernel (148 SMs x 2 blocks x 512 threads)
YEAR_DRIFT_STEPS = 8640          # one model day
YEAR_TIMED_STEPS = 640
YEAR_REBIN_THRESHOLD = 0.03      # re-bin when more than 3 % of the lane-layers of a launch were idle
# --dump-outputs: per-column outputs of every column up to DUMP_COLUMNS (a seeded sample beyond), layer profiles of a
# seeded sample of DUMP_PROFILE_COLUMNS columns; together at most DUMP_MAX_BYTES
DUMP_COLUMNS = 1 << 20
DUMP_PROFILE_COLUMNS = 1024
DUMP_PROFILES = ["m", "S_abs", "H_abs", "thick", "T"]
DUMP_MAX_BYTES = 64 * 10**6


def load_state(rec: int) -> dict:
    z = np.load(ROOT / "tests" / "golden" / "sheba_oracle_states.npz")
    p = f"state{rec}_"
    return {k[len(p):]: (z[k] if z[k].ndim else z[k].item()) for k in z.files if k.startswith(p)}


def load_sites(nrec_min: int) -> np.ndarray:
    z = np.load(ROOT / "tests" / "golden" / "forcing_era.npz")
    n = min(z[s].shape[1] for s in SITES)
    assert n >= nrec_min
    return np.stack([z[s][:, :n] for s in SITES])  # [9, 4, n]


def _perturbation_block(b: int):
    """The five perturbation vectors of global columns [b*TOTAL_COLUMNS, (b+1)*TOTAL_COLUMNS)."""
    # drawn per block of TOTAL_COLUMNS so that a column's numbers do not depend on the sharding; block 0 is the
    # config-5 ensemble (default_rng(4), SURVEY 8d), further blocks extend it for the weak-scaling runs
    rng = np.random.default_rng(4) if b == 0 else np.random.default_rng([4, b])
    T2m_off = rng.uniform(-2, 2, TOTAL_COLUMNS)
    lw = rng.uniform(0.95, 1.05, TOTAL_COLUMNS)
    sw = rng.uniform(0.9, 1.1, TOTAL_COLUMNS)
    pr = rng.uniform(0.5, 1.5, TOTAL_COLUMNS)
    amp = 7.0 * rng.uniform(0.5, 1.5, TOTAL_COLUMNS)
    return T2m_off, lw, sw, pr, amp


def perturbations(col0: int, n: int):
    """Deterministic per-column perturbations for global columns [col0, col0+n)."""
    scale = np.ones((4, n))
    offset = np.zeros((4, n))
    amp = np.empty(n)
    done = 0
    while done < n:
        g = col0 + done
        b, lo = divmod(g, TOTAL_COLUMNS)
        cnt = min(n - done, TOTAL_COLUMNS - lo)
        T2m_off, lw, sw, pr, am = _perturbation_block(b)
        sl, dst = slice(lo, lo + cnt), slice(done, done + cnt)
        scale[0, dst], scale[1, dst], scale[3, dst] = sw[sl], lw[sl], pr[sl]
        offset[2, dst] = T2m_off[sl]
        amp[dst] = am[sl]
        done += cnt
    site = (np.arange(col0, col0 + n) % len(SITES)).astype(np.int32)
    return site, scale, offset, amp


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self) -> dict:
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 3 + j and r[3 + j].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def make_oracle_columns(st: dict, sites: np.ndarray, cols: np.ndarray, backend: str = "det"):
    from oracle import oracle
    out = []
    for c in cols:
        s, sc, of, am = perturbations(int(c), 1)
        col = oracle.Column(4, backend)
        col.set_forcing(*[sites[s[0], k] * sc[k, 0] + of[k, 0] for k in range(4)])
        col.load_state(st)
        col.set_scalar("oflux_amp", float(am[0]))
        out.append(col)
    return out


def cpu_oracle_rate(st: dict, sites: np.ndarray, ncols: int, nsteps: int, nthreads: int, reps: int = 1, backend: str = "libm"):
    """column-steps/s of the CPU oracle, one column per OS thread."""
    from oracle import oracle
    oracle.build()
    cols = make_oracle_columns(st, sites, np.linspace(0, TOTAL_COLUMNS - 1, ncols).astype(np.int64), backend)
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        rc = oracle.run_batch(cols, nsteps, nthreads)
        times.append(time.perf_counter() - t0)
        if rc:
            raise RuntimeError(f"oracle STOP {rc}")
    return ncols * nsteps / min(times), times


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on all host cores.  The Fortran cannot
    be compiled here, so this is the oracle port in its libm build (the math library the reference binary links)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncores = os.cpu_count() or 1
    st = load_state(START_RECORD)
    sites = load_sites(64)
    sample_cols = 4 * ncores
    from oracle import oracle
    oracle.build()
    idx = np.linspace(0, TOTAL_COLUMNS - 1, sample_cols).astype(np.int64)
    cols = make_oracle_columns(st, sites, idx, "libm")
    steps_per = MODEL_STEPS * 64  # 4,096 model steps per bench step: a few seconds of CPU work on all host cores
    for _ in range(args.warmup):
        oracle.run_batch(cols, steps_per, ncores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rc = oracle.run_batch(cols, steps_per, ncores)
        if rc:
            raise RuntimeError(f"oracle STOP {rc}")
    dt = time.perf_counter() - t0
    value = sample_cols * steps_per * args.steps / dt
    # the deterministic-math build (what the GPU is compared with bit for bit), one bench step, for the record
    cols_det = make_oracle_columns(st, sites, idx, "det")
    t0 = time.perf_counter()
    oracle.run_batch(cols_det, steps_per, ncores)
    value_det = sample_cols * steps_per / (time.perf_counter() - t0)
    per = args.columns if args.scaling == "weak" else args.columns // max(args.gpus, 1)
    line = {
        "impl": "reference", "metric": "column-timesteps/sec (FP64, 100 layers)", "value": value,
        "unit": "column-timesteps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus, scaling=args.scaling, per_gpu=per),
        "cpu_baseline": {"value": value, "unit": "column-timesteps/s", "cores": ncores, "kind": "port",
                         "sample": f"{sample_cols} of the {per * max(args.gpus, 1)} columns x {steps_per} model steps per bench step "
                                   f"({steps_per * args.steps} timed), one column per thread; C oracle, libm build "
                                   "(gcc -O2 -ffp-contract=off), the Fortran reference cannot be compiled in this image",
                         "det_build_value": value_det},
        "e2e": {"value": value, "unit": "column-timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(n_gpus: int, scaling: str = "weak", per_gpu: int | None = None) -> dict:
    per = per_gpu if per_gpu is not None else (TOTAL_COLUMNS if scaling == "weak" else TOTAL_COLUMNS // n_gpus)
    cfg = {
        "workload": "config 5: 1,048,576 ERA-interim-style columns per GPU (testcase 4 flags, Nlayer 100, dt 10 s), "
                    "mid-January SHEBA state (N_active 100, snow 0.124 m), per-column perturbed forcing of 9 sites",
        "columns_total": per * n_gpus, "columns_per_gpu": per,
        "model_steps_per_step": MODEL_STEPS, "layers": 100, "dt_s": 10.0,
        "parallelism": f"columns sharded over {n_gpus} GPU(s), no data-path collective",
        "cache": "working set (>= 12 KB/column x columns) is far larger than the 126 MB L2; no flush needed",
    }
    return cfg


def make_engine(api, st: dict, sites: np.ndarray, per: int, col0: int, device: int):
    """`per` columns of the ensemble starting at global column col0, all in state `st`, with their own forcing."""
    cfg = api.Config.from_state({**st, "thick_min": st["thick_min"]})
    eng = api.Engine(cfg, per, device)
    eng.load_column_state(st, 0)
    eng.broadcast_column(0, 0, per)
    site, scale, offset, amp = perturbations(col0, per)
    eng.set_forcing(sites, site, scale, offset)
    eng.set_scalar("oflux_amp", amp)
    return eng


def year_weighted(api, sites: np.ndarray, device: int) -> dict:
    """Throughput over the regimes of a SHEBA year (see the module docstring)."""
    rows, t_per_step = [], 0.0
    # the ERA-interim site files hold one year (2,920 three-hourly records); the late-summer state lies in the second
    # year of the run, so the annual cycle of every site is repeated once
    sites = np.concatenate([sites[:, :, :2920], sites[:, :, :2920]], axis=2)
    for rec, what, share in YEAR_REGIMES:
        eng = make_engine(api, load_state(rec), sites, YEAR_COLUMNS, 0, device)
        # re-binning is driven by the divergence the kernel measures itself (idle lane-layers per warp), checked
        # between calls: the drift runs in eight calls of three model hours
        eng.set_rebin_auto(YEAR_REBIN_THRESHOLD)
        for _ in range(YEAR_DRIFT_STEPS // 1080):
            eng.step(1080)
        eng.step(YEAR_TIMED_STEPS // 2)        # warm
        eng.step(YEAR_TIMED_STEPS, sync=False)
        eng.synchronize()
        ms = eng.last_step_ms()
        rate = YEAR_COLUMNS * YEAR_TIMED_STEPS / (ms * 1e-3)
        na = eng.get_int("N_active")
        div = eng.divergence()
        rows.append({"record": rec, "regime": what, "share": share, "value": rate, "N_active_mean": float(na.mean()),
                     "N_active_min": int(na.min()), "N_active_max": int(na.max()), "failed_columns": int(eng.count_failed()),
                     "idle_lane_layer_share": div["idle_lane_layer_share"], "snow_class_split_warp_share": div["snow_class_split_warp_share"],
                     "rebins": div["rebins"]})
        t_per_step += share / rate
        eng.close()
    return {"value": 1.0 / t_per_step, "unit": "column-timesteps/s", "columns": YEAR_COLUMNS, "drift_steps": YEAR_DRIFT_STEPS,
            "timed_steps": YEAR_TIMED_STEPS, "rebin": f"automatic, kernel-measured idle lane-layer share > {YEAR_REBIN_THRESHOLD}", "regimes": rows,
            "how": "harmonic mean of the regime rates weighted by the regime's share of the golden SHEBA records"}


def column_sample(n: int, k: int, seed: int) -> np.ndarray:
    """All n columns if n <= k, else a fixed seeded sample of k of them, in increasing order."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def dump_outputs(out_dir: str, eng, diag_names: list, diag: np.ndarray, red: dict) -> None:
    """Write the outputs of the last timed step as out_dir/<name>.npy (see the module docstring)."""
    cols = column_sample(eng.ncol, DUMP_COLUMNS, 0)
    out = {name: diag[j, cols] for j, name in enumerate(diag_names)}
    out["ensemble_reduction"] = np.array([[v["sum"], v["min"], v["max"]] for v in red.values()])  # rows in reduce_diag order
    for name in ("N_active", "status"):
        out[name] = eng.get_int(name)[cols].astype(np.float32)
    if len(cols) < eng.ncol:
        out["columns"] = cols.astype(np.float64)
    pcols = column_sample(eng.ncol, DUMP_PROFILE_COLUMNS, 1)
    out["profile_columns"] = pcols.astype(np.float64)
    for name in DUMP_PROFILES:
        out[f"profile_{name}"] = np.concatenate([eng.get_array(name, int(c), 1) for c in pcols])
    nbytes = sum(a.nbytes for a in out.values())
    assert nbytes <= DUMP_MAX_BYTES, nbytes
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(d / f"{name}.npy", a)


def main():
    global MODEL_STEPS
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--columns", type=int, default=TOTAL_COLUMNS,
                    help="columns per GPU (weak scaling, default: the config-5 ensemble) or in total (--scaling strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-year-weighted", action="store_true", help="skip the six-regime year-weighted block (N = 1 only)")
    ap.add_argument("--two-pass", action="store_true", help="kernel tuning: the two-pass step (samsim_step_kernel<true>) instead of the general path")
    ap.add_argument("--model-steps", type=int, default=MODEL_STEPS, help="model timesteps per bench step (one launch)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: samsim_b200 has no CPU path (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: NCCL prints its version banner (and, with NCCL_DEBUG set, its log) to
        # stdout when the communicator is created, i.e. at the first collective -- do that with fd 1 pointing at stderr
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    from samsim_b200 import api, distributed as D

    if args.scaling == "weak":   # per-GPU work fixed: rank r owns global columns [r*per, (r+1)*per)
        per = args.columns
        col0, total = rank * per, per * world
    else:                        # total fixed, contiguous shards
        total = args.columns
        col0, per = D.shard(total, rank, world)
    st = load_state(START_RECORD)
    sites = load_sites(64)
    MODEL_STEPS = args.model_steps
    eng = make_engine(api, st, sites, per, col0, local_rank)
    eng.set_tuning(args.two_pass)
    eng.set_snapshot_mode(api.SNAP_SCALARS_ONLY)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- FP64 peak of this GPU (live) ----
    fp64_peak = api.fp64_peak(local_rank, 1.2)

    # ---- warm-up ----
    for _ in range(max(args.warmup, 3)):
        eng.step(MODEL_STEPS)

    # ---- timed region A: device-resident ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    l0 = eng.launch_count()
    kernel_ms = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.step(MODEL_STEPS, sync=False)
        eng.synchronize()
        kernel_ms += eng.last_step_ms()     # CUDA events on the launching stream
    barrier()
    wall_a = time.perf_counter() - t0
    launches = eng.launch_count() - l0

    # ---- timed region B: end to end through the C ABI with host buffers ----
    # every step: upload this step's forcing table from pinned host memory, advance, read back the step's result:
    # five per-column diagnostics (ice thickness, bulk salinity, freeboard, snow depth, surface temperature) into
    # pinned host memory + the 18-number ensemble reduction
    DIAG = ["thickness", "bulk_salin", "freeboard", "thick_snow", "T_top"]
    pinned_in = torch.from_numpy(np.ascontiguousarray(sites)).pin_memory()
    pinned_out = torch.empty((len(DIAG), per), dtype=torch.float64).pin_memory()
    diag_host = pinned_out.numpy()
    h2d = pinned_in.numel() * 8
    d2h = diag_host.nbytes + 18 * 8
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.update_forcing(pinned_in.numpy())
        eng.step(MODEL_STEPS, sync=False)
        for j, name in enumerate(DIAG):
            eng.get_scalar(name, 0, per, out=diag_host[j])
        red = eng.reduce_diag()
    barrier()
    wall_b = time.perf_counter() - t0
    assert np.isfinite(diag_host).all() and red["N_active"]["max"] <= 100
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, DIAG, diag_host, red)

    # ---- ensemble diagnostics: the only cross-GPU exchange of the model (NCCL all-reduce of 18 numbers) ----
    ensemble = D.reduce_ensemble(eng.reduce_diag(), per, device=torch.device("cuda", local_rank))
    nf = torch.tensor([eng.count_failed()], dtype=torch.int64, device="cuda")

    # ---- strong scaling: the SAME 1,048,576-column ensemble sharded over the ranks (fixed total) ----
    strong = None
    if world > 1 and args.scaling == "weak":
        eng.close()
        s_col0, s_per = D.shard(TOTAL_COLUMNS, rank, world)
        eng_s = make_engine(api, st, sites, s_per, s_col0, local_rank)
        for _ in range(max(args.warmup, 3)):
            eng_s.step(MODEL_STEPS)
        barrier()
        t0 = time.perf_counter()
        ms_s = 0.0
        for _ in range(args.steps):
            eng_s.step(MODEL_STEPS, sync=False)
            eng_s.synchronize()
            ms_s += eng_s.last_step_ms()
        barrier()
        wall_s = time.perf_counter() - t0
        ts = torch.tensor([ms_s * 1e-3, wall_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        strong = {"columns_total": TOTAL_COLUMNS, "columns_per_gpu": int(s_per), "value": TOTAL_COLUMNS * MODEL_STEPS * args.steps / float(ts[1]),
                  "kernel_value": TOTAL_COLUMNS * MODEL_STEPS * args.steps / float(ts[0]), "unit": "column-timesteps/s",
                  "ms_per_step": float(ts[1]) / args.steps * 1e3,
                  "note": "fixed total: the config-5 ensemble split over the ranks; no data-path collective"}
        eng = eng_s

    # ---- max over ranks ----
    t = torch.tensor([kernel_ms * 1e-3, wall_a, wall_b], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(nf, op=dist.ReduceOp.SUM)
    kern_s, wall_a_s, wall_b_s = [float(x) for x in t.tolist()]
    col_steps = total * MODEL_STEPS * args.steps
    value = col_steps / wall_a_s
    kernel_rate = col_steps / kern_s

    if rank == 0:
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        per_gpu_rate = kernel_rate / world
        achieved_tf = per_gpu_rate * F_ALG_FLOP_PER_COLUMN_STEP / 1e12
        # DRAM traffic of the step kernel from the committed ncu capture (profiles/): bytes per column-step there,
        # scaled to the columns x steps of one launch here (None if the digest is missing)
        traffic, traffic_src = None, None
        try:
            dig = json.loads((ROOT / "profiles" / NCU_DIGEST).read_text())
            m = dig["metrics"]
            unit = {"Gbyte": 1e9, "Mbyte": 1e6, "Tbyte": 1e12, "Kbyte": 1e3, "byte": 1.0}
            dram = sum(float(m[k][0]) * unit[m[k][1]] for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
            per_colstep = dram / NCU_DIGEST_COLUMN_STEPS
            traffic = per_colstep * per * MODEL_STEPS
            traffic_src = (f"profiles/{NCU_DIGEST}: {per_colstep / 1e3:.1f} KB of DRAM traffic per column-step (ncu --set full, "
                           f"{NCU_DIGEST_COLUMN_STEPS} column-steps in the captured launch) x the column-steps of one launch here")
            # FP64 pipe instructions per column-step (thread level) from the same capture -> the pipe's issue ceiling
            cyc = float(m["sm__cycles_elapsed.max"][0])
            pc = {op: float(m[f"smsp__sass_thread_inst_executed_op_{op}_pred_on.sum.per_cycle_elapsed"][0]) for op in ("dadd", "dmul", "dfma")}
            fp64_inst = sum(pc.values()) * cyc / NCU_DIGEST_COLUMN_STEPS
            hw_flop = (pc["dadd"] + pc["dmul"] + 2.0 * pc["dfma"]) * cyc / NCU_DIGEST_COLUMN_STEPS
        except Exception:
            fp64_inst = hw_flop = None
        clocks = sampler.summary()
        issue = None
        if fp64_inst:
            sm_hz = (clocks.get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)) * 1e6
            ceiling = 148 * 64 * sm_hz / fp64_inst
            issue = {"fp64_inst_per_column_step": fp64_inst, "ceiling": ceiling, "unit": "column-timesteps/s",
                     "frac": per_gpu_rate / ceiling, "hw_flop_per_column_step": hw_flop,
                     "how": "148 SMs x 64 FP64 lanes x sampled SM clock / FP64 instructions per column-step (dadd + dmul + dfma, "
                            f"profiles/{NCU_DIGEST}); with -fmad=false a multiply-add is two pipe slots, so the DFMA peak is not reachable"}
        line = {
            "metric": "column-timesteps/sec (FP64, 100 layers)", "value": value, "unit": "column-timesteps/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": wall_a_s / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(world, scaling=args.scaling, per_gpu=per),
            "kernel_path": "two-pass step (samsim_step_kernel<true>)" if args.two_pass else "general path (samsim_step_kernel<false>)",
            "e2e": {"value": col_steps / wall_b_s, "unit": "column-timesteps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "fp64", "achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac": achieved_tf / fp64_peak, "traffic": traffic, "traffic_unit": "bytes of DRAM traffic per launch",
                         "traffic_source": traffic_src,
                         "peak_source": "DFMA micro-benchmark on this GPU in this run (samsim_b200_fp64_peak); MEASURED_PEAKS.json has no FP64 entry",
                         "flop_per_column_step": F_ALG_FLOP_PER_COLUMN_STEP,
                         "flop_note": "operation count of the reference algorithm AS WRITTEN (oracle counting build); the kernel "
                                      "skips work bit-identically (lazy freezing point, S4 sweep reuse, O(N) sums), so `achieved` is an "
                                      "algorithmic rate; hw_tflops is what the hardware executed",
                         "hw_tflops": (per_gpu_rate * hw_flop / 1e12) if hw_flop else None,
                         "issue_ceiling": issue,
                         "kernel": "samsim_step_kernel", "kernel_ms_per_launch": kern_s / max(launches, 1) * 1e3,
                         "hbm": {"achieved": per_gpu_rate * B_ALG_BYTES_PER_COLUMN_STEP / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": per_gpu_rate * B_ALG_BYTES_PER_COLUMN_STEP / 1e9 / hbm_peak,
                                 "bytes_per_column_step": B_ALG_BYTES_PER_COLUMN_STEP,
                                 # what the kernel really moves (ncu traffic per launch / measured launch time): the second limit
                                 "dram_gbs": (traffic / (kern_s / max(launches, 1)) / 1e9) if traffic else None,
                                 "dram_frac": (traffic / (kern_s / max(launches, 1)) / 1e9 / hbm_peak) if traffic else None,
                                 "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650 GB/s"}},
            "clocks": clocks,
            "failed_columns": int(nf.item()),
            "ensemble": {k: ensemble[k] for k in ("thickness", "thick_snow", "N_active", "columns")},
        }
        if strong is not None:
            line["strong"] = strong
        if world == 1 and not args.no_year_weighted:
            eng.close()
            line["year_weighted"] = year_weighted(api, sites, local_rank)
        if world == 1 and not args.no_cpu_baseline:
            ncores = os.cpu_count() or 1
            ncols_cpu, nsteps_cpu = 4 * ncores, 50000   # ~10 s of CPU work on all host cores
            rate, times = cpu_oracle_rate(st, sites, ncols_cpu, nsteps_cpu, ncores, backend="libm")
            line["cpu_baseline"] = {"value": rate, "unit": "column-timesteps/s", "cores": ncores, "kind": "port",
                                    "sample": f"{ncols_cpu} of the {total} columns x {nsteps_cpu} model steps, one column per thread "
                                              f"({times[0]:.1f} s); C oracle in its libm build, Fortran reference not compilable here"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
