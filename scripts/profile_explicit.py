"""Throughput, HBM traffic and latency of the explicit Runge-Kutta kernel (csrc/erk_batch.cu: RK23, DOP853) next to the
on-chip RK45 kernel, in one GPU call:

  * the card's name and power limit (part of every number below);
  * throughput: 4096-column lattice (sweep_lattice(default, 16, 16, 16)), N = 200, events on, launches of a fixed
    budget of step attempts resumed from the device state as bench.py does, timed with CUDA events after a warm-up:
    step attempts/s and RHS evaluations/s per method, and the new kernel's algorithmic HBM bytes (erk_algorithmic_bytes)
    against the copy bandwidth measured in the same run;
  * single-column latency: the default scenario to t = 0.03 with events (RK23, DOP853, RK45);
  * RK23 sweep to T*: the 4096 columns in predicted_cost order, events on, to t = 1.

    python scripts/profile_explicit.py [attempts per launch] [timed launches] [T* wall limit s]
Prints one JSON document."""
import json
import os
import subprocess
import sys
import time
from dataclasses import asdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "integrating-diagenetic-equations-using-python_b200"))
import ctypes as C  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402

import marlpde_b200 as mb  # noqa: E402
from marlpde_b200 import _cabi, batch  # noqa: E402
from marlpde.parameters import Map_Scenario  # noqa: E402


def erk_algorithmic_bytes(method, n_cells, attempts, accepted, dense_steps, launches_x_columns, events=True):
    """HBM bytes the explicit kernel moves by construction (csrc/erk_batch.cu; every vector in the per-column workspace,
    V = 5 N doubles; a zero tableau coefficient skips its row):
      stage s            stage input y + h sum_j a_sj K_j (read y and the K_j with a_sj != 0, write 1 V), RHS (read
                         1 V, write 1 V)
      y_new              read y and the K_j with b_j != 0, write 1 V; f(y_new) 2 V
      error norm         read y, y_new and the K_j with a non-zero error weight
      accepted step      event predicate bits of y_new (1 V) when events are on
      dense output       DOP853: the three extra stages, like stage s, in the steps that sample t_eval or locate events
      column start       f(y) once per launch (2 V) and the state copy in and out (2 V)"""
    from scipy.integrate._ivp.rk import DOP853, RK23
    M = RK23 if method == "RK23" else DOP853
    V = 5.0 * n_cells * 8.0
    A = np.asarray(M.A)
    stages = sum(np.count_nonzero(A[s, :s]) + 4 for s in range(1, M.n_stages))
    ynew = np.count_nonzero(M.B) + 2 + 2
    E = np.asarray(M.E) if method == "RK23" else (np.asarray(M.E3) != 0) | (np.asarray(M.E5) != 0)
    err = 2 + np.count_nonzero(E)
    per_attempt = (stages + ynew + err) * V
    extra = 0.0
    if method == "DOP853":
        AX = np.asarray(M.A_EXTRA)
        extra = sum(np.count_nonzero(AX[i, :M.n_stages + 1 + i]) + 4 for i in range(AX.shape[0])) * V
    return (attempts * per_attempt + accepted * (V if events else 0.0) + dense_steps * extra
            + launches_x_columns * 4 * V)


def device_info():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,power.max_limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        out["nvidia_smi"] = q
    except (OSError, subprocess.TimeoutExpired):
        out["nvidia_smi"] = "unavailable"
    return out


def copy_bandwidth_gbs(nbytes=2 << 30, reps=10):
    a = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    b.copy_(a)
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e-3)
    del a, b
    return 2 * nbytes / best / 1e9


class Stepper:
    """Budgeted launches on device buffers, resumed from the device state (bench.py's RK45 stepper, any method)."""

    def __init__(self, method, P, y0, attempts, evcap=16, t_bound=1.0):
        self.method, self.lib = method, _cabi.lib()
        self.B, self.N = y0.shape[0], y0.shape[2]
        dev = torch.device("cuda", 0)
        self.d_params = batch.params_to_device(P, dev)
        self.d_y = torch.from_numpy(y0).to(dev)
        self.d_state = torch.from_numpy(batch.make_state(self.B, 0.0, 1e-6).view(np.uint8).copy()).to(dev)
        self.d_ec = torch.zeros((self.B, 7), dtype=torch.int32, device=dev)
        self.d_et = torch.full((self.B, 7, evcap), float("nan"), dtype=torch.float64, device=dev)
        if method == "RK45":
            self.d_queue = torch.zeros(1 + 2 * self.B, dtype=torch.int32, device=dev)
            flags = _cabi.FLAG_EVENTS | _cabi.FLAG_QUEUE_LOCKS
        else:
            self.d_queue = torch.zeros(1, dtype=torch.int32, device=dev)
            self.nb = int(getattr(self.lib, f"marlpde_{method.lower()}_workspace_bytes")(self.B, self.N))
            self.d_work = torch.empty(self.nb // 8 + 1, dtype=torch.float64, device=dev)
            flags = _cabi.FLAG_EVENTS
        self.opts = _cabi.RK45Options(t_bound=t_bound, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=attempts,
                                      n_eval=0, event_capacity=evcap, flags=flags, quantum=0)
        self.stream = torch.cuda.current_stream()

    def state(self):
        return self.d_state.cpu().numpy().view(_cabi.STATE_DTYPE)

    def step(self):
        self.d_queue.zero_()
        s = self.stream.cuda_stream
        if self.method == "RK45":
            _cabi.check(self.lib.marlpde_rk45_integrate_dev(
                self.d_y.data_ptr(), self.d_params.data_ptr(), self.d_state.data_ptr(), self.B, self.N, C.byref(self.opts),
                None, None, self.d_ec.data_ptr(), self.d_et.data_ptr(), self.d_queue.data_ptr(), s))
        else:
            _cabi.check(getattr(self.lib, f"marlpde_{self.method.lower()}_integrate_dev")(
                self.d_y.data_ptr(), self.d_params.data_ptr(), self.d_state.data_ptr(), self.B, self.N, C.byref(self.opts),
                None, None, self.d_ec.data_ptr(), self.d_et.data_ptr(), self.d_work.data_ptr(), self.nb,
                self.d_queue.data_ptr(), s))


def throughput(method, P, y0, attempts, launches):
    st = Stepper(method, P, y0, attempts)
    st.step()                                                   # warm-up launch (module load, first budget)
    torch.cuda.synchronize()
    s0 = st.state().copy()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(launches)]
    for e0, e1 in ev:
        e0.record(st.stream)
        st.step()
        e1.record(st.stream)
    torch.cuda.synchronize()
    secs = sum(a.elapsed_time(b) for a, b in ev) * 1e-3
    s1 = st.state()
    att = int((s1["n_accepted"] + s1["n_rejected"]).sum() - (s0["n_accepted"] + s0["n_rejected"]).sum())
    acc = int(s1["n_accepted"].sum() - s0["n_accepted"].sum())
    nfev = int(s1["nfev"].sum() - s0["nfev"].sum())
    out = {"method": method, "columns": st.B, "n_cells": st.N, "attempts_per_launch": attempts, "launches": launches,
           "seconds": secs, "attempts": att, "rhs_evaluations": nfev, "attempts_per_s": att / secs,
           "rhs_evaluations_per_s": nfev / secs, "finished_columns": int((s1["status"] == 0).sum())}
    if method != "RK45":
        stages = 3 if method == "RK23" else 12
        dense = (nfev - st.B * launches - stages * att) // 3 if method == "DOP853" else 0
        out["algorithmic_bytes"] = erk_algorithmic_bytes(method, st.N, att, acc, dense, st.B * launches)
        out["algorithmic_gbs"] = out["algorithmic_bytes"] / secs / 1e9
    return out


def latency(method, pde):
    run = {"RK23": mb.integrate_rk23_batch, "DOP853": mb.integrate_dop853_batch, "RK45": mb.integrate_rk45_batch}[method]
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    y = torch.from_numpy(y0).cuda()
    run(y, P, t_span=(0, 1e-4), first_step=1e-6)                # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = run(y, P, t_span=(0, 0.03), first_step=1e-6, t_eval=[0.0, 0.03], events=True, event_capacity=32)
    e1.record()
    torch.cuda.synchronize()
    return {"method": method, "seconds": e0.elapsed_time(e1) * 1e-3, "nfev": int(r.nfev[0]),
            "attempts": int(r.n_attempts[0]), "status": int(r.status[0]), "event_counts": r.event_counts[0].tolist()}


def sweep_to_tstar(method, pde, wall_limit, budget=200_000):
    order = np.argsort(-mb.sweep.predicted_cost(pde, method), kind="stable")
    P, y0 = mb.derive_column_params(pde)[order], mb.initial_state(pde)[order]
    st = Stepper(method, P, y0, budget)
    torch.cuda.synchronize()
    w0 = time.time()
    launches = 0
    while True:
        st.step()
        launches += 1
        s = st.state()                                          # synchronises
        if not np.any(s["status"] == 1) or time.time() - w0 > wall_limit:
            break
    secs = time.time() - w0
    return {"method": method, "columns": st.B, "order": "predicted_cost, longest first", "seconds": secs,
            "launches_of_budget": [launches, budget], "finished": int((s["status"] == 0).sum()),
            "step_too_small": int((s["status"] == -1).sum()), "unfinished": int((s["status"] == 1).sum()),
            "attempts": int((s["n_accepted"] + s["n_rejected"]).sum()), "rhs_evaluations": int(s["nfev"].sum()),
            "t_min": float(s["t"].min())}


def main():
    attempts = int(sys.argv[1]) if len(sys.argv) > 1 else 400
    launches = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    wall = float(sys.argv[3]) if len(sys.argv) > 3 else 420.0
    base = asdict(Map_Scenario())
    lat = mb.sweep_lattice(base, 16, 16, 16)
    P, y0 = mb.derive_column_params(lat), mb.initial_state(lat)
    doc = {"device": device_info(), "copy_bandwidth_gbs": copy_bandwidth_gbs()}
    doc["throughput"] = [throughput(m, P, y0, attempts, launches) for m in ("RK23", "DOP853", "RK45")]
    for t in doc["throughput"]:
        if "algorithmic_gbs" in t:
            t["hbm_roofline_share"] = t["algorithmic_gbs"] / doc["copy_bandwidth_gbs"]
    print(json.dumps(doc["throughput"]), file=sys.stderr, flush=True)
    doc["single_column_latency"] = [latency(m, base) for m in ("RK23", "DOP853", "RK45")]
    print(json.dumps(doc["single_column_latency"]), file=sys.stderr, flush=True)
    doc["sweep_to_tstar"] = sweep_to_tstar("RK23", lat, wall)
    doc["sweep_to_tstar"]["rk45_reference_seconds"] = 131.4
    print(json.dumps(doc, indent=1))


if __name__ == "__main__":
    main()
