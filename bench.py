#!/usr/bin/env python
"""bench.py — column RK-steps/s of the batched RK45 integrator and time-to-T* (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--no-tstar] [--no-large-n]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1], SURVEY.md §8d config 2): the synthetic 4096-column
Map_Scenario parameter sweep (16 x 16 x 16 lattice over sedimentation rate, b, D0co3), N=200
depth cells, RK45 rtol=atol=1e-3, first_step=1e-6.  One bench "step" = every column of the sweep
advances by `--attempts` adaptive RK45 step attempts (each attempt = 6 RHS evaluations + stage
algebra + error norm) in ONE launch of the persistent kernel, resuming where the previous step
stopped; the concatenation of steps is the integration to T*.  At N>1 GPUs every rank owns
8192 columns of the 32x32x64 lattice (65,536 columns at 8 GPUs, configs[2]); no collective on
the data path, one NCCL all-gather of the end states after the timed steps.

`value`  = step attempts of all columns / device time, inputs resident in HBM (CUDA events).
`e2e`    = same through the host-pointer C-ABI call (marlpde_rk45_integrate) with pinned HOST
           buffers: H2D of state+params, kernel, D2H of state, every step.
`roofline` is fp64-pipe based: achieved = value x 307,600 algorithmic flop per column-step
           (SURVEY.md §8d) against an fp64 FMA peak measured on the same device in this run.
`equal_load` (N=1 only): the headline step repeated with 8192 columns, the per-GPU load of the
           N>1 runs, so that the per-GPU rate of an N-GPU run can be compared at equal load.
`time_to_Tstar` (the second half of BASELINE's metric; on by default): the whole sweep from t=0 to T* with
           the RK45 kernel (N=1 only, ~2 min) and with the implicit Radau kernel (both scenario bases; at N>1 the
           8192-columns-per-GPU sweep with the cost-balanced column assignment and the all-gather of the
           snapshots timed), each with its own roofline block and a CPU figure beside it.
`bdf_time_to_Tstar` (N=1): the same sweep with the variable-order BDF kernel (method="BDF"; LSODA's stiff mode), HBM
           roofline from its own byte model, SciPy BDF on the host cores beside it.
`large_n_streaming` (N=1): the streaming / overlapped-tile RK45 path at N = 2 000 / 20 000 with fp64 and HBM rooflines.
`cpu_baseline` / `--impl reference`: the reference's own path — SciPy solve_ivp(RK45) driving the
           restated numba RHS (oracle/, kind "port": py-pde is not installable here) — on the
           host cores of the same box, one column per process, bounded sample.
`--dump-outputs DIR` writes what the headline step returned after the last timed step as DIR/<name>.npy (float64; see
           dump_outputs), so that two builds run with the same arguments can be compared output for output.

The benchmark writes nothing into the source tree: no bytecode, and numba's cache goes to a temporary directory.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "integrating-diagenetic-equations-using-python_b200")
sys.path.insert(0, PKG)

FLOP_PER_COLUMN_STEP_PER_CELL = 1538          # SURVEY.md §8d: N*(6*198 + 5*70)
METRIC = "column RK-steps/sec at N=200"
UNIT = "column-steps/s"
HBM_PEAK_FALLBACK_GBS = 6550.4                # MEASURED_PEAKS.json of this pool (copy bandwidth)


def scenario_base(name: str) -> dict:
    """asdict(Map_Scenario()) values (marlpde/parameters.py:16-143) via the host mirror."""
    from marlpde.parameters import Map_Scenario
    from dataclasses import asdict
    base = asdict(Map_Scenario())
    if name == "scenario_A":
        base |= {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    return base


def lattice_for(world: int):
    return (16, 16, 16) if world == 1 else (32, 32, 64)


def hbm_peak_gbs():
    """(GB/s, source) — MEASURED_PEAKS.json when the driver wrote one, else the pool's documented figure."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy bandwidth)"
    except (OSError, ValueError, KeyError):
        return HBM_PEAK_FALLBACK_GBS, "fallback: 6550.4 GB/s (B200_PROFILING.md / last MEASURED_PEAKS.json of this pool)"


# --------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def summary(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.rows:
            if ts < t0 - 0.1 or ts > t1 + 0.1:
                continue
            p = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(p[0]))
                smax = float(p[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- CPU reference arm
def _cpu_worker(job):
    """One column, SciPy RK45 on the restated numba RHS (what Evolve_scenario.py:104-109 does)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import lheureux_oracle as oracle
    pde, t_end, warm = job
    if warm:                                     # JIT compile outside the timed call
        oracle.integrate(pde, method="RK45", t_span=(0.0, 1e-5), t_eval=[0.0, 1e-5], events=False)
    t0 = time.perf_counter()
    sol = oracle.integrate(pde, method="RK45", first_step=1e-6, rtol=1e-3, atol=1e-3, t_span=(0.0, t_end),
                           t_eval=np.array([0.0, t_end]), events=True)
    return (sol.nfev - 1) // 6, time.perf_counter() - t0, sol.status


def _cpu_radau_worker(job):
    """One column to T* the way the reference's default Solver() does it (parameters.py:207-221): SciPy Radau,
    rtol = atol = 1e-3, first_step 1e-6, the reference's jac_sparsity, the 7 event monitors."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import lheureux_oracle as oracle
    pde, warm = job[0], job[1]
    method = job[2] if len(job) > 2 else "Radau"
    n = int(pde["N"])
    sp = oracle.jacobian_sparsity(n)
    if warm:
        oracle.integrate(pde, method=method, t_span=(0.0, 1e-5), t_eval=[0.0, 1e-5], events=False, jac_sparsity=sp)
        return 0.0, 0, 0, 0, 0
    t0 = time.perf_counter()
    try:
        sol = oracle.integrate(pde, method=method, first_step=1e-6, rtol=1e-3, atol=1e-3, t_span=(0.0, 1.0),
                               t_eval=np.array([0.0, 1.0]), events=True, jac_sparsity=sp)
        return time.perf_counter() - t0, int(sol.status), int(sol.nfev), int(sol.njev), int(sol.nlu)
    except (FloatingPointError, ZeroDivisionError, ValueError):
        return time.perf_counter() - t0, -9, 0, 0, 0


def _lattice_columns(base_name: str, count: int, spread: bool = False):
    import numpy as np
    import marlpde_b200 as mb
    pde = mb.sweep_lattice(scenario_base(base_name), 16, 16, 16)
    idx = np.linspace(0, 4095, count).round().astype(int) if spread else np.arange(count)
    return [{k: (float(v[c]) if np.ndim(v) else v) for k, v in pde.items()} for c in idx]


def cpu_reference_pass(base_name: str, t_end: float, cores: int, pool, warm: bool):
    """First `cores` columns of the sweep lattice, one process each, integrated to t_end."""
    jobs = [(one, t_end, warm) for one in _lattice_columns(base_name, cores)]
    t0 = time.perf_counter()
    res = pool.map(_cpu_worker, jobs)
    wall = time.perf_counter() - t0
    attempts = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    return attempts, busy, wall


def cpu_radau_pass(base_name: str, cores: int, pool, method: str = "Radau"):
    """`cores` columns spread over the lattice, SciPy Radau (or BDF) to T*, one process each: seconds per column."""
    cols = _lattice_columns(base_name, cores, spread=True)
    pool.map(_cpu_radau_worker, [(c, True, method) for c in cols])                       # JIT + first touch
    res = pool.map(_cpu_radau_worker, [(c, False, method) for c in cols])
    secs = [r[0] for r in res]
    return {"seconds_per_column_mean": sum(secs) / len(secs), "seconds_per_column_max": max(secs),
            "columns_sampled": len(cols), "finished": sum(1 for r in res if r[1] == 0), "cores": cores,
            "seconds_per_4096_columns_on_these_cores": sum(secs) / len(secs) * 4096 / cores, "kind": "port",
            "nfev_mean": sum(r[2] for r in res) / len(res), "njev_mean": sum(r[3] for r in res) / len(res),
            "nlu_mean": sum(r[4] for r in res) / len(res),
            "sample": f"SciPy solve_ivp({method}, rtol=atol=1e-3, first_step=1e-6, reference jac_sparsity, 7 events) on the numba "
                      "RHS (oracle port), columns spread evenly over the 16x16x16 lattice, one process per core, full T*"}


def run_reference_arm(args, rank: int, world: int):
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    ctx = mp.get_context("fork")
    t_end = args.cpu_t_end
    with ctx.Pool(cores) as pool:
        cpu_reference_pass(args.base, 1e-4, cores, pool, warm=True)             # compile + warm-up
        for _ in range(max(args.warmup - 1, 0)):
            cpu_reference_pass(args.base, t_end / 10, cores, pool, warm=False)
        tot_att, tot_t = 0, 0.0
        for _ in range(args.steps):
            att, busy, _wall = cpu_reference_pass(args.base, t_end, cores, pool, warm=False)
            tot_att += att
            tot_t += busy
    value = tot_att / tot_t
    sample = (f"first {cores} columns of the 16x16x16 lattice ({args.base} base), SciPy solve_ivp RK45 + numba RHS "
              f"(oracle port), t in [0,{t_end}] of T*, {tot_att // args.steps} step attempts per pass, one process per core")
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": workload_config(args, world),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_config(args, world: int) -> dict:
    lat = lattice_for(world)
    per_gpu = 4096 if world == 1 else 8192
    return {"workload": (f"{per_gpu * world}-column Map_Scenario sweep ({'one column in every %d of the ' % (8 // world) if 1 < world < 8 else ''}{lat[0]}x{lat[1]}x{lat[2]} lattice over "
                         f"sedimentationrate, b, D0co3; {args.base} base), N=200, RK45 rtol=atol=1e-3, "
                         f"first_step=1e-6; {args.attempts} step attempts per column per bench step, resumed"),
            "columns": per_gpu * world, "columns_per_gpu": per_gpu, "n_cells": 200,
            "attempts_per_column_per_step": args.attempts, "parallelism": f"columns sharded x{world}, no data-path collective",
            "scaling_note": ("weak scaling, 8192 columns per GPU at N>1; BASELINE's 1-GPU config is 4096 columns, so the N=1 line "
                             "also carries `equal_load` = the same step with 8192 columns: compare per-GPU rates against that"),
            "l2_policy": "256 MiB buffer written between timed steps (L2 flush); state is shared-memory resident"}


def strided_selection(n_all: int, world: int):
    """8192 columns per GPU taken as every (8/world)-th column of the 65,536-column lattice, so that every world
    size covers the full parameter ranges (world = 8: the whole lattice)."""
    import numpy as np
    stride = max(1, n_all // (8192 * world))
    return np.arange(0, n_all, stride)[: 8192 * world]


# --------------------------------------------------------------------------- GPU arm, pieces
class Rk45Stepper:
    """Device-resident columns advanced by `attempts` step attempts per call through the device-pointer C ABI."""

    def __init__(self, P, y0, attempts, dev, evcap=16):
        import ctypes as C
        import numpy as np
        import torch
        from marlpde_b200 import _cabi, batch
        self.C, self.np, self.torch, self._cabi = C, np, torch, _cabi
        self.lib = _cabi.lib()
        self.B, self.N = y0.shape[0], y0.shape[2]
        self.P = P
        self.d_params = batch.params_to_device(P, dev)
        self.d_y = torch.from_numpy(y0).to(dev)
        self.d_state = torch.from_numpy(batch.make_state(self.B, 0.0, 1e-6).view(np.uint8).copy()).to(dev)
        self.d_queue = torch.zeros(1 + 2 * self.B, dtype=torch.int32, device=dev)   # counter + lock + attempts words
        self.d_ec = torch.zeros((self.B, 7), dtype=torch.int32, device=dev)
        self.evcap = evcap
        self.d_et = torch.full((self.B, 7, evcap), float("nan"), dtype=torch.float64, device=dev)
        # the 7 event monitors run inside the timed region, as in the reference's solve_ivp call
        # (Evolve_scenario.py:107-109 passes events=[...]); roots are located and stored (first evcap per monitor)
        self.opts = _cabi.RK45Options(t_bound=1.0, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=attempts,
                                      n_eval=0, event_capacity=evcap, flags=_cabi.FLAG_EVENTS | _cabi.FLAG_QUEUE_LOCKS,
                                      quantum=0)
        self.stream = torch.cuda.current_stream()

    def state(self):
        return self.d_state.cpu().numpy().view(self._cabi.STATE_DTYPE)

    def attempts_done(self):
        st = self.state()
        return int(st["n_accepted"].sum() + st["n_rejected"].sum())

    def step(self, opts=None):
        self.d_queue.zero_()
        o = self.opts if opts is None else opts
        self._cabi.check(self.lib.marlpde_rk45_integrate_dev(
            self.d_y.data_ptr(), self.d_params.data_ptr(), self.d_state.data_ptr(), self.B, self.N, self.C.byref(o),
            None, None, self.d_ec.data_ptr(), self.d_et.data_ptr(), self.d_queue.data_ptr(), self.stream.cuda_stream))


def timed_steps(stepper, steps, flush, barrier):
    import torch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    a0 = stepper.attempts_done()
    barrier()
    w0 = time.time()
    for s in range(steps):
        ev[s][0].record(stepper.stream)
        stepper.step()
        ev[s][1].record(stepper.stream)
        flush.fill_(s & 1)                                          # L2 flush between timed steps (not timed)
    barrier()
    w1 = time.time()
    a1 = stepper.attempts_done()
    return a1 - a0, sum(a.elapsed_time(b) for a, b in ev), w0, w1


DUMP_BUDGET_BYTES = 64_000_000


def dump_outputs(out_dir, stepper, rank, world):
    """What the headline step hands its caller, as float64 .npy files: the column states `y` [B, 5, N], the per-column
    integrator records `state_*` (t, h_abs, step counts, nfev, status), the event monitors' `event_counts` [B, 7] and
    `event_times`: the located roots only, min(count, evcap) of them per column and monitor, concatenated in
    (column, monitor) order (the kernel fills slots from 0 and leaves the rest of the NaN-filled buffer untouched).
    `column_index` says which columns of this rank's block were written: all of them when they fit
    DUMP_BUDGET_BYTES with every event slot filled (4096 columns at N=200: 37 MB at most), else a sample drawn
    with a fixed seed.
    At N>1 GPUs every rank writes its own block, file names suffixed with _rank<r>."""
    import numpy as np
    st = stepper.state()
    per_column = 8 * (5 * stepper.N + 7 + 7 * stepper.evcap + 7)
    keep = min(stepper.B, DUMP_BUDGET_BYTES // world // per_column)
    cols = np.arange(stepper.B)
    if keep < stepper.B:
        cols = np.sort(np.random.default_rng(0).choice(stepper.B, keep, replace=False))
    counts = stepper.d_ec.cpu().numpy()[cols]
    located = np.arange(stepper.evcap) < np.minimum(counts, stepper.evcap)[..., None]
    arrays = {"column_index": cols, "y": stepper.d_y.cpu().numpy()[cols],
              "event_counts": counts, "event_times": stepper.d_et.cpu().numpy()[cols][located]}
    for field in ("t", "h_abs", "n_accepted", "n_rejected", "nfev", "status"):
        arrays["state_" + field] = st[field][cols]
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def radau_algorithmic_bytes(n_cells, newton, nlu, njev, steps_attempted):
    """HBM bytes the implicit kernel has to move by construction (DESIGN.md §5): all per-column vectors, Jacobian
    blocks and fp32 records live in a per-column HBM workspace.  V = 5 N doubles (one state-sized vector).
      Newton iteration   3 stage evaluations (read y + Z_s, write F_s: 9 V), B = TI F - M W (read 6 V, write 3 V),
                         block-tridiagonal solve of both systems (two sweeps: read and write B, 3 V each way, plus the
                         fp32 records 2 x 408 B per cell), norm / W += dW / Z = T W pass (read 7 V, write 6 V)
      factorisation pair read the Jacobian blocks (600 B per cell), write the records (512 B per cell)
      Jacobian           analytic blocks in one pass: read y (1 V), write 600 B per cell
      step attempt       Z0 / W start values (read 5 V, write 6 V), error estimate (read 4 V, write 2 V, one real solve:
                         2 V + 2 x 204 B per cell), commit (read 4 V, write 5 V), f(y_new) (2 V)"""
    V = 5.0 * n_cells * 8.0
    per_newton = 9 * V + 9 * V + (12 * V + 2 * 408.0 * n_cells) + 13 * V
    per_lu_pair = (600.0 + 512.0) * n_cells
    per_jac = V + 600.0 * n_cells
    per_step = 11 * V + (6 * V + 2 * V + 2 * 204.0 * n_cells) + 9 * V + 2 * V
    return newton * per_newton + (nlu / 2.0) * per_lu_pair + njev * per_jac + steps_attempted * per_step


def bdf_algorithmic_bytes(n_cells, newton, nlu, njev, steps_attempted, rescalings):
    """HBM bytes the BDF kernel has to move by construction (csrc/bdf_batch.cu; V = 5 N doubles):
      Newton iteration   residual b = M (c f(y) - psi - d) fused into the RHS pass (read y, psi, d, write b: 4 V), real
                         block-tridiagonal solve (two sweeps: read and write b, 4 V, plus the compact fp32 records
                         2 x 208 B per cell), norm / y += dy / d += dy pass (read 3 V, write 2 V)
      factorisation      read the Jacobian blocks (600 B per cell), write the compact record (308 B per cell)
      Jacobian           analytic blocks in one pass: read y (1 V), write 600 B per cell
      step attempt       predictor y = sum D, psi, d = 0 (read ~4 V of D at the typical order 3, write 3 V), error norm
                         (read 2 V), differences update (read ~6 V, write ~6 V)
      rescaling          change_D: read and write order + 1 ~ 4 rows of D (8 V)"""
    V = 5.0 * n_cells * 8.0
    per_newton = 4 * V + (4 * V + 2 * 208.0 * n_cells) + 5 * V
    per_lu = (600.0 + 308.0) * n_cells
    per_jac = V + 600.0 * n_cells
    per_step = 7 * V + 2 * V + 12 * V
    return newton * per_newton + nlu * per_lu + njev * per_jac + steps_attempted * per_step + rescalings * 8 * V


def implicit_sweep(mb, batch, torch, dev, sw_pde, columns, evcap=16, t_eval=None, method="Radau"):
    """The implicit kernel on `columns` of the sweep dictionary, t = 0 .. T*; returns (result, seconds)."""
    import numpy as np
    Pi = mb.derive_column_params(sw_pde)[columns]
    yi = mb.initial_state(sw_pde)[columns]
    d_yi = torch.from_numpy(np.ascontiguousarray(yi)).to(dev)
    d_pi = batch.params_to_device(np.ascontiguousarray(Pi), dev)
    torch.cuda.synchronize()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.current_stream()
    r0.record(stream)
    run = mb.integrate_radau_batch if method == "Radau" else mb.integrate_bdf_batch
    rr = run(d_yi, d_pi, t_span=(0.0, 1.0), first_step=1e-6, rtol=1e-3, atol=1e-3,
             events=True, event_capacity=evcap, inplace=True, t_eval=t_eval)
    r1.record(stream)
    torch.cuda.synchronize()
    return rr, r0.elapsed_time(r1) * 1e-3


def implicit_block(rr, secs, n_cells, peak_gbs, peak_src, method="Radau"):
    import numpy as np
    attempts = float(rr.n_accepted.sum() + rr.n_rejected.sum() + rr.newton_failures.sum())
    if method == "Radau":
        alg = radau_algorithmic_bytes(n_cells, float(rr.newton_iterations.sum()), float(rr.nlu.sum()),
                                      float(rr.njev.sum()), attempts)
    else:   # bdf.py: a rescaling of D after every rejection / Newton failure and after about every fourth accepted step
        alg = bdf_algorithmic_bytes(n_cells, float(rr.newton_iterations.sum()), float(rr.nlu.sum()), float(rr.njev.sum()),
                                    attempts, float(rr.n_rejected.sum() + rr.newton_failures.sum()) + 0.25 * float(rr.n_accepted.sum()))
    kernel = "radau_kernel" if method == "Radau" else "bdf_kernel"
    return {"method": ("Radau IIA (radau_kernel, one launch)" if method == "Radau"
                       else "variable-order BDF = SciPy BDF step for step; LSODA's stiff mode (bdf_kernel, one launch)"),
            "seconds": secs, "columns": int(rr.status.shape[0]), "finished": int((rr.status == 0).sum()),
            "status_histogram": {str(int(k)): int(v) for k, v in zip(*np.unique(rr.status, return_counts=True))},
            "steps_per_column_min_max": [int(rr.n_accepted.min()), int(rr.n_accepted.max())],
            "radau_steps": int(rr.n_accepted.sum()), "rejected": int(rr.n_rejected.sum()),
            "newton_iterations": int(rr.newton_iterations.sum()), "newton_failures": int(rr.newton_failures.sum()),
            "lu_factorisations": int(rr.nlu.sum()), "jacobians": int(rr.njev.sum()), "nfev": int(rr.nfev.sum()),
            "radau_steps_per_s": float(rr.n_accepted.sum() + rr.n_rejected.sum()) / secs,
            "roofline": {"bound": "hbm", "achieved": alg / secs / 1e9, "peak": peak_gbs, "unit": "GB/s",
                         "frac": alg / secs / 1e9 / peak_gbs, "traffic": None, "kernel": kernel,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
                         "algorithmic_bytes_per_step_attempt": alg / max(attempts, 1.0),
                         "traffic_note": "dram bytes of this launch are not measured in-run (ncu: profiles/)"}}


def run_gpu_arm(args, rank: int, local_rank: int, world: int):
    import numpy as np
    import torch
    import marlpde_b200 as mb
    from marlpde_b200 import _cabi, batch, sweep
    import ctypes as C

    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _cabi.lib()

    lat = lattice_for(world)
    pde = mb.sweep_lattice(scenario_base(args.base), *lat)
    if world > 1:
        sel = strided_selection(lat[0] * lat[1] * lat[2], world)
        pde = sweep.shard(pde, sel)
    P_all = mb.derive_column_params(pde)
    y_all = mb.initial_state(pde)
    a, b = sweep.partition(P_all.shape[0], world)[rank]
    sl = slice(a, b)                                              # contiguous column block per rank
    P, y0 = P_all[sl], y_all[sl]
    B, N = y0.shape[0], y0.shape[2]
    EVCAP = 16
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    stepper = Rk45Stepper(P, y0, args.attempts, dev, EVCAP)
    for _ in range(args.warmup):
        stepper.step()
        flush.fill_(1)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    att_dev, dev_ms, w0, w1 = timed_steps(stepper, args.steps, flush, barrier)
    st = stepper.state()
    kernel_ms = dev_ms / args.steps
    clocks = sampler.summary(w0, w1) if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, stepper, rank, world)

    # ---- e2e: the host-pointer C-ABI call with pinned host buffers, copies inside the timed region
    h_y = torch.from_numpy(stepper.d_y.cpu().numpy()).pin_memory()
    h_state = torch.from_numpy(st.view(np.uint8).copy()).pin_memory()
    h_params = torch.from_numpy(P.view(np.uint8).copy()).pin_memory()
    h_ec = torch.zeros((B, 7), dtype=torch.int32).pin_memory()
    h_et = torch.full((B, 7, EVCAP), float("nan"), dtype=torch.float64).pin_memory()
    hy, hs, hp, hec, het = h_y.numpy(), h_state.numpy(), h_params.numpy(), h_ec.numpy(), h_et.numpy()
    e2e_steps = max(2, args.steps)

    def e2e_step():
        _cabi.check(lib.marlpde_rk45_integrate(hy.ctypes.data, hp.ctypes.data, hs.ctypes.data, B, N, C.byref(stepper.opts),
                                               None, None, hec.ctypes.data, het.ctypes.data, local_rank))
    e2e_step()                                                       # warm-up (allocations, first touch)
    barrier()
    sview = hs.view(_cabi.STATE_DTYPE)
    b0 = int(sview["n_accepted"].sum() + sview["n_rejected"].sum())
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    b1 = int(sview["n_accepted"].sum() + sview["n_rejected"].sum())
    h2d = hy.nbytes + hp.nbytes + hs.nbytes + hec.nbytes + het.nbytes
    d2h = hy.nbytes + hs.nbytes + hec.nbytes + het.nbytes

    # ---- aggregate over ranks: max time, sum of work; one all-gather of end states (the only collective)
    att = torch.tensor([att_dev, b1 - b0], dtype=torch.float64, device=dev)
    tms = torch.tensor([dev_ms, e2e_s, w1 - w0], dtype=torch.float64, device=dev)
    gather_ms = None
    if dist is not None:
        dist.all_reduce(att, op=dist.ReduceOp.SUM)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        out = torch.empty((world * B, 5, N), dtype=torch.float64, device=dev)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        g0.record()
        dist.all_gather_into_tensor(out, stepper.d_y)
        g1.record()
        torch.cuda.synchronize()
        gather_ms = g0.elapsed_time(g1)
        del out
    total_attempts, e2e_attempts = float(att[0]), float(att[1])
    dev_s, e2e_s, wall_s = float(tms[0]) * 1e-3, float(tms[1]), float(tms[2])
    value = total_attempts / dev_s

    # ---- roofline: fp64 FMA peak measured on this device, now
    peak = C.c_double(0.0)
    _cabi.check(lib.marlpde_probe_fp64_peak(local_rank, 4096, 5, C.byref(peak)))
    hbm_gbs, hbm_src = hbm_peak_gbs()
    line = None
    if rank == 0:
        flop_per_launch = (total_attempts / world / args.steps) * FLOP_PER_COLUMN_STEP_PER_CELL * N
        achieved = flop_per_launch / (kernel_ms * 1e-3) / 1e12
        roof = {"bound": "fp64", "achieved": achieved, "peak": peak.value, "unit": "TFLOP/s",
                "frac": achieved / peak.value if peak.value else None, "traffic": None,
                "peak_source": "measured in this run: marlpde_probe_fp64_peak (8 independent DFMA chains/thread, "
                               "2048 threads/SM, best of 5); MEASURED_PEAKS.json has no fp64 entry",
                "algorithmic_flop_per_column_step": FLOP_PER_COLUMN_STEP_PER_CELL * N,
                "kernel": "rk45_persistent_kernel", "kernel_ms_per_launch": kernel_ms,
                "hbm_bytes_per_launch_algorithmic": 2 * B * 5 * N * 8}
        prof = os.path.join(ROOT, "profiles", "roofline_latest.json")
        if os.path.exists(prof):
            try:
                with open(prof) as fh:
                    pj = json.load(fh)
                roof["traffic"] = pj.get("dram_bytes_per_launch")
                roof["traffic_source"] = ("NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one "
                                          "`ncu --set full` capture, " + str(pj.get("source", "profiles/roofline_latest.json")))
            except (OSError, ValueError):
                pass
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(args, world),
                "e2e": {"value": e2e_attempts / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": e2e_steps, "api": "marlpde_rk45_integrate (host pointers, pinned)"},
                "gpu_launches": args.steps, "roofline": roof, "clocks": clocks,
                "per_gpu_value": value / world,
                "wall_s_timed_region": wall_s, "t_reached_min_max": [float(st["t"].min()), float(st["t"].max())],
                "accepted_rejected": [int(st["n_accepted"].sum()), int(st["n_rejected"].sum())]}
        if gather_ms is not None:
            line["allgather_end_states_ms"] = gather_ms

    # ---- N = 1: the same step at the per-GPU load of the multi-GPU runs (8192 columns)
    if world == 1 and not args.no_equal_load:
        big = mb.sweep_lattice(scenario_base(args.base), 32, 32, 64)
        big = sweep.shard(big, strided_selection(32 * 32 * 64, 1))
        s2 = Rk45Stepper(mb.derive_column_params(big), mb.initial_state(big), args.attempts, dev, EVCAP)
        for _ in range(3):
            s2.step()
            flush.fill_(1)
        n2 = max(3, min(args.steps, 5))
        att2, ms2, _, _ = timed_steps(s2, n2, flush, barrier)
        line["equal_load"] = {"columns_per_gpu": s2.B, "value": att2 / (ms2 * 1e-3), "unit": UNIT, "steps": n2,
                              "what": "same bench step with 8192 columns (every 8th column of the 32x32x64 lattice), the "
                                      "per-GPU load of the N>1 runs: per-GPU rate at N GPUs / this = scaling efficiency at "
                                      "equal load"}
        del s2

    tstar = not args.no_tstar
    # ---- time-to-T* with the explicit kernel (N = 1): whole sweep, longest columns first
    if tstar and world == 1 and not args.skip_rk45_tstar:
        order = np.argsort(-sweep.predicted_cost(pde) * np.ones(B), kind="stable")      # longest first: short tail
        s3 = Rk45Stepper(np.ascontiguousarray(P[order]), np.ascontiguousarray(y0[order]), args.step_cap, dev, EVCAP)
        # Columns that reach T* need 0.50-1.18 M attempts on this lattice.  A few columns run into a singularity
        # of the model near t = 0.5-0.7 and end with status -1 (step below 10 ulp, as SciPy does); how many
        # attempts they burn there is chaotic (0.7-6.8 M seen for the same column in two builds that differ by
        # FMA contraction only) and a lone column advances at ~50 k attempts/s, so the cap bounds the tail.
        # (columns longest first, claimed whole; only the last 2 x 444 — the shortest — are cut into quanta so that the
        #  slots do not run dry one by one over the ~9 s the last whole column would take.  Cutting all columns into
        #  quanta makes them advance in lock-step and leaves the longest ones alone at the end: 151 s instead of 138 s.)
        o2 = _cabi.RK45Options(t_bound=1.0, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=args.step_cap, n_eval=0,
                               event_capacity=EVCAP,
                               flags=_cabi.FLAG_EVENTS | _cabi.FLAG_QUEUE_LOCKS | _cabi.FLAG_QUEUE_TAIL, quantum=0)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        f0.record(s3.stream)
        s3.step(o2)
        f1.record(s3.stream)
        torch.cuda.synchronize()
        st2 = s3.state()
        secs = f0.elapsed_time(f1) * 1e-3
        tot = int(st2["n_accepted"].sum() + st2["n_rejected"].sum())
        flops = float(tot) * FLOP_PER_COLUMN_STEP_PER_CELL * N
        line["time_to_Tstar"] = {
            "method": "RK45 (rk45_persistent_kernel, one launch, columns longest first, the last 888 cut into quanta)",
            "seconds": secs, "columns": B, "step_attempts": tot, "column_steps_per_s": tot / secs,
            "step_cap_per_column": args.step_cap, "finished": int((st2["status"] == 0).sum()),
            "status_histogram": {str(int(k)): int(v) for k, v in zip(*np.unique(st2["status"], return_counts=True))},
            "events_located_per_monitor": s3.d_ec.cpu().numpy().sum(axis=0).tolist(),
            "unfinished_columns": [[int(order[c]), int(st2["status"][c]), float(st2["t"][c]), float(st2["h_abs"][c])]
                                   for c in np.nonzero(st2["status"] != 0)[0][:32]],
            "steps_per_column_min_max": [int((st2["n_accepted"] + st2["n_rejected"]).min()),
                                         int((st2["n_accepted"] + st2["n_rejected"]).max())],
            "roofline": {"bound": "fp64", "achieved": flops / secs / 1e12, "peak": peak.value, "unit": "TFLOP/s",
                         "frac": flops / secs / 1e12 / peak.value if peak.value else None, "traffic": None,
                         "kernel": "rk45_persistent_kernel",
                         "algorithmic_flop_per_column_step": FLOP_PER_COLUMN_STEP_PER_CELL * N}}
        del s3

    # ---- time-to-T* with the implicit kernel (BASELINE.json configs[4]); N > 1: cost-balanced shards + all-gather
    if tstar:
        implicit = {}
        t_eval = np.array([0.0, 1.0])
        # warm-up: first launch of the implicit kernel (module load) on a handful of columns, not timed
        mb.integrate_radau_batch(torch.from_numpy(np.ascontiguousarray(y0[:8])).to(dev), P[:8], t_span=(0.0, 1e-3),
                                 first_step=1e-6, events=True, event_capacity=EVCAP)
        for base_name in ("scenario_A", "default"):
            sw = mb.sweep_lattice(scenario_base(base_name), *lat)
            assign, nB = None, B
            if world > 1:
                sw = sweep.shard(sw, strided_selection(lat[0] * lat[1] * lat[2], world))
                nB = sweep.n_columns_of(sw)
                cost_i = sweep.predicted_cost(sw, "Radau") * np.ones(nB)
                assign = sweep.balanced_assignment(cost_i, world)
                mine = assign[rank]
                mine = mine[np.argsort(-cost_i[mine], kind="stable")]
            else:
                # columns are claimed from a queue in batch order: longest first by the a-priori cost estimate of the
                # implicit path (sweep.predicted_cost: 21.2 s in lattice order, 18.3 s in this order, 17.9-18.5 s when
                # ordered by the work MEASURED in a previous sweep — the estimate leaves nothing on the table)
                mine = np.argsort(-sweep.predicted_cost(sw, "Radau") * np.ones(B), kind="stable")
            barrier()
            rr, secs = implicit_sweep(mb, batch, torch, dev, sw, mine, EVCAP, t_eval=t_eval)
            blk = implicit_block(rr, secs, N, hbm_gbs, hbm_src)
            if dist is not None:
                # the one collective of the sweep: snapshots [B/G, 2, 5, N] of every rank to every rank
                tt = torch.tensor([secs], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                cnt = torch.tensor([blk["radau_steps"] + blk["rejected"], blk["finished"], blk["newton_iterations"],
                                    blk["lu_factorisations"], blk["jacobians"],
                                    blk["roofline"]["algorithmic_bytes_per_launch"]], dtype=torch.float64, device=dev)
                dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                g0.record()
                snaps = sweep.gather_columns(rr.snapshots, [len(x) for x in assign])
                g1.record()
                torch.cuda.synchronize()
                gms = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device=dev)
                dist.all_reduce(gms, op=dist.ReduceOp.MAX)
                per_gpu_gbs = float(cnt[5]) / float(tt[0]) / 1e9 / world
                blk = {"method": blk["method"], "seconds": float(tt[0]), "columns": int(nB), "columns_per_gpu": int(len(mine)),
                       "finished": int(cnt[1]), "radau_step_attempts": int(cnt[0]), "newton_iterations": int(cnt[2]),
                       "lu_factorisations": int(cnt[3]), "jacobians": int(cnt[4]),
                       "assignment": "sweep.balanced_assignment (columns sorted by predicted cost, dealt out boustrophedon)",
                       "allgather_snapshots_ms": float(gms[0]), "allgather_bytes": int(snaps.numel() * 8),
                       "rank0": blk,
                       "roofline": {"bound": "hbm", "achieved": per_gpu_gbs, "peak": hbm_gbs, "unit": "GB/s per GPU",
                                    "frac": per_gpu_gbs / hbm_gbs, "traffic": None, "kernel": "radau_kernel",
                                    "peak_source": hbm_src}}
                del snaps
            implicit[base_name] = blk
            del rr
        if rank == 0:
            line["implicit_time_to_Tstar"] = implicit
        if world == 1 and not args.no_bdf:
            # the other implicit solver of the reference (method="BDF"; LSODA's stiff mode): same sweep, same order
            mb.integrate_bdf_batch(torch.from_numpy(np.ascontiguousarray(y0[:8])).to(dev), P[:8], t_span=(0.0, 1e-3),
                                   first_step=1e-6, events=True, event_capacity=EVCAP)
            sw = mb.sweep_lattice(scenario_base("default"), *lat)
            mine = np.argsort(-sweep.predicted_cost(sw, "BDF") * np.ones(B), kind="stable")
            rb, secs = implicit_sweep(mb, batch, torch, dev, sw, mine, EVCAP, t_eval=t_eval, method="BDF")
            line["bdf_time_to_Tstar"] = {"default": implicit_block(rb, secs, N, hbm_gbs, hbm_src, method="BDF")}
            del rb

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- large depth grids (BASELINE.json configs[3]): streaming RK45, fp64 and HBM rooflines
    if world == 1 and not args.no_large_n:
        large = {}
        stream = torch.cuda.current_stream()
        for nL, bL, attL in ((20000, 64, 96), (2000, 64, 256), (20000, 1, 256)):
            pL = scenario_base("scenario_A") | {"N": nL}
            PL = np.repeat(mb.derive_column_params(pL), bL)
            yL = torch.from_numpy(np.repeat(mb.initial_state(pL), bL, 0)).to(dev)
            dPL = batch.params_to_device(PL, dev)
            stL = batch.make_state(bL, 0.0, 1e-6 * (200 / nL) ** 2)
            d_stL = torch.from_numpy(stL.view(np.uint8).copy()).to(dev)
            nb = int(lib.marlpde_rk45_stream_workspace_bytes(bL, nL))
            d_wL = torch.empty(nb // 8 + 1, dtype=torch.float64, device=dev)
            oL = _cabi.RK45Options(t_bound=1.0, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=attL, n_eval=0,
                                   event_capacity=0, flags=0, quantum=0)

            def run_large():
                _cabi.check(lib.marlpde_rk45_stream_integrate_dev(yL.data_ptr(), dPL.data_ptr(), d_stL.data_ptr(), bL, nL,
                                                                  C.byref(oL), None, None, d_wL.data_ptr(), nb,
                                                                  stream.cuda_stream))
            run_large()                                            # warm-up (also moves past the first steps)
            torch.cuda.synchronize()
            l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0.record(stream)
            run_large()
            l1.record(stream)
            torch.cuda.synchronize()
            secs = l0.elapsed_time(l1) * 1e-3
            tiles_mode = os.environ.get("MARLPDE_RK45_STREAM", "tiles")[0] != "s"
            # algorithmic HBM bytes per cell and attempt: overlapped tiles read y, K1 and write y_new, K7
            # (4 vector passes x 40 B; y ping-pongs between two buffers); one launch per stage moves 42 passes
            per_cell = 160.0 if tiles_mode else 1680.0
            alg_bytes = per_cell * nL * bL * attL
            flops = FLOP_PER_COLUMN_STEP_PER_CELL * float(nL) * bL * attL
            large[f"N{nL}_B{bL}"] = {
                "n_cells": nL, "columns": bL, "attempts_per_column": attL, "seconds": secs,
                "mode": "overlapped tiles (1 launch per attempt)" if tiles_mode else "1 launch per stage",
                "column_steps_per_s": bL * attL / secs, "cell_steps_per_s": bL * attL * nL / secs,
                "working_set_MB": nb / 1e6, "launches": (2 if tiles_mode else 7) * attL + 4,
                "roofline": {"bound": "fp64" if tiles_mode else "hbm", "achieved": flops / secs / 1e12, "peak": peak.value,
                             "unit": "TFLOP/s", "frac": flops / secs / 1e12 / peak.value if peak.value else None,
                             "traffic": None, "kernel": "tile_attempt_kernel" if tiles_mode else "stage kernels"},
                "roofline_hbm": {"bound": "hbm", "achieved": alg_bytes / secs / 1e9, "peak": hbm_gbs, "unit": "GB/s",
                                 "frac": alg_bytes / secs / 1e9 / hbm_gbs, "traffic": None, "peak_source": hbm_src,
                                 "algorithmic_bytes_per_cell_attempt": per_cell}}
            del yL, d_wL
        line["large_n_streaming"] = large

    if world == 1 and not args.no_cpu_baseline:
        import multiprocessing as mp
        cores = os.cpu_count() or 1
        with mp.get_context("fork").Pool(cores) as pool:
            cpu_reference_pass(args.base, 1e-4, cores, pool, warm=True)
            catt, cbusy, _ = cpu_reference_pass(args.base, args.cpu_t_end, cores, pool, warm=False)
            line["cpu_baseline"] = {
                "value": catt / cbusy, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": (f"first {cores} columns of the lattice, SciPy solve_ivp RK45 + numba RHS (oracle port of the "
                           f"reference path; py-pde not installable), t in [0,{args.cpu_t_end}] of T*, {catt} step attempts, "
                           f"one process per core, {cbusy:.1f} s")}
            if "time_to_Tstar" in line:
                line["time_to_Tstar"]["cpu_seconds_extrapolated"] = line["time_to_Tstar"]["step_attempts"] / (catt / cbusy)
                line["time_to_Tstar"]["cpu_note"] = (f"the sweep's step attempts at the CPU port's measured rate on {cores} "
                                                     "cores (cpu_baseline.value)")
            if tstar and not args.no_cpu_radau:
                for base_name in ("scenario_A", "default"):
                    line["implicit_time_to_Tstar"][base_name]["cpu_baseline"] = cpu_radau_pass(base_name, cores, pool)
                if "bdf_time_to_Tstar" in line:
                    line["bdf_time_to_Tstar"]["default"]["cpu_baseline"] = cpu_radau_pass("default", cores, pool, "BDF")
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--base", default="default", choices=["default", "scenario_A"])
    ap.add_argument("--attempts", type=int, default=3000, help="RK45 step attempts per column per bench step")
    ap.add_argument("--full", action="store_true", help="(kept for compatibility: everything is on by default now)")
    ap.add_argument("--no-tstar", action="store_true", help="skip the time-to-T* sweeps (RK45 ~2 min, implicit ~25 s)")
    ap.add_argument("--no-large-n", action="store_true", help="skip the N = 2 000 / 20 000 streaming lines")
    ap.add_argument("--no-equal-load", action="store_true", help="N=1: skip the 8192-column repeat of the headline step")
    ap.add_argument("--step-cap", type=int, default=2_000_000,
                    help="step-attempt cap per column of the RK45 sweep to T* (SURVEY.md 8d, config 2: 'give every "
                         "column a step cap + status'); 0 = none")
    ap.add_argument("--skip-rk45-tstar", action="store_true",
                    help="time-to-T* without the ~140 s explicit sweep (implicit sweep only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cpu-radau", action="store_true", help="skip the SciPy Radau sample beside the implicit sweep")
    ap.add_argument("--no-bdf", action="store_true", help="N=1: skip the BDF sweep to T* (~20 s + its SciPy BDF sample)")
    ap.add_argument("--cpu-t-end", type=float, default=0.03, help="CPU sample: integrate to this fraction of T*")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline step's outputs after the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    # the tree may be read-only: no bytecode next to the sources, numba's cache (oracle/, cache=True) elsewhere
    sys.dont_write_bytecode = True
    os.environ.setdefault("NUMBA_CACHE_DIR", os.path.join(tempfile.gettempdir(), f"marlpde-bench-numba-{os.getuid()}"))
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
    else:
        run_gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
