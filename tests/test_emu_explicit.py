"""The explicit Runge-Kutta kernel (csrc/erk_batch.cu: RK23, DOP853) compiled for the host and run by the SIMT emulator
(tests/emu/, see test_emu_kernels.py), against live SciPy on the oracle RHS.  Test infrastructure, not a CPU path of the
product: this checks the stage loop, step control, error norms, dense output, event location and budget / resume logic
of the kernel before it runs on a GPU.

Precision of the comparison.  RK23 reproduces SciPy to round-off (1e-15).  DOP853's error estimate cancels about five
orders of magnitude (|K| ~ 2e5 on this RHS against |K^T E5| ~ 1.6 in the first step), so the summation order of the
estimate — the kernel's fma chain against the BLAS dgemv SciPy calls — moves the error norm in its 11th digit and the
next step size in its 10th.  With the same accept / reject decisions that leaves the end states 5e-11 apart over the
short horizons here (measured), and t_eval samples inside a step up to 8e-9 apart: the stiff modes sit at the stability
limit of the method, where the seventh-order interpolant of a step is sensitive to its length (the interpolation formula
itself agrees with SciPy's Dop853DenseOutput to 5e-16 on the same stages).  The DOP853 state gate is therefore 2e-8; nfev
is still identical."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
from scipy.integrate import solve_ivp

import lheureux_oracle as oracle
import marlpde_b200 as mb
from marlpde_b200 import _cabi, batch
from conftest import ROOT

EMU = os.path.join(ROOT, "tests", "emu")
SCEN_A = {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
METHODS = {"RK23": 0, "DOP853": 1}
STATE_GATE = {"RK23": 1e-12, "DOP853": 2e-8}
np.seterr(all="ignore")


@pytest.fixture(scope="module")
def emu_erk():
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    out = os.path.join(EMU, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemu_erk.so")
    srcs = [os.path.join(EMU, f) for f in ("emu_erk.cc", "simt_emu.cc")]
    done = subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-DMARLPDE_HOST_EMU", "-I", EMU, "-o", so] + srcs,
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    assert done.returncode == 0, done.stdout.decode()
    lib = C.CDLL(so)
    lib.emu_erk.restype = C.c_int

    def run(method, P, y, t_end, t_eval=(), events=False, first_step=1e-6, max_steps=0, state=None, flags=0,
            counts=None, times=None):
        y = np.ascontiguousarray(y, dtype=np.float64).copy()
        P = np.ascontiguousarray(P)
        B, _, N = y.shape
        st = batch.make_state(B, 0.0, first_step) if state is None else state.copy()
        te = np.asarray(t_eval, dtype=np.float64)
        snap = np.full((B, max(1, te.size), 5, N), np.nan)
        ec = np.zeros((B, 7), np.int32) if counts is None else counts.copy()
        et = np.full((B, 7, 16), np.nan) if times is None else times.copy()
        o = _cabi.RK45Options(t_bound=t_end, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=max_steps,
                              n_eval=te.size, event_capacity=16,
                              flags=flags | (_cabi.FLAG_EVENTS if events else 0), quantum=0)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = lib.emu_erk(METHODS[method], p(y), p(P), p(st), B, N, C.byref(o), p(te), p(snap), p(ec), p(et))
        assert rc == 0, f"emulated {method} kernel: rc {rc} (deadlock or mismatched collective, see stderr)"
        return dict(y=y, state=st, snapshots=snap, event_counts=ec, event_times=et)
    return run


def event_start(n_cells=200):
    """Scenario A with a few cells pushed across monitor thresholds: four monitors fire within the first steps."""
    pde = oracle.default_scenario() | SCEN_A | {"N": n_cells}
    y0 = mb.initial_state(pde)
    for f, frac, v in ((0, 0.25, -2e-5), (1, 0.30, -1e-5), (4, 0.75, 1.0 + 5e-6)):
        y0[:, f, int(frac * n_cells)] = v
    return pde, y0


@pytest.mark.parametrize("method", ["RK23", "DOP853"])
def test_explicit_kernel_under_emulation_is_scipy_step_for_step(emu_erk, method):
    """Scenario A over a short horizon with t_eval samples (t0 included): the same nfev, accepted and rejected steps as
    SciPy, end state and samples within the gate of the module docstring."""
    pde = oracle.default_scenario() | SCEN_A
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    t_end = 2e-4
    te = [0.0, 0.7e-4, 1.3e-4, t_end]
    sol = oracle.integrate(pde, method=method, t_span=(0, t_end), t_eval=te, events=False, first_step=1e-6)
    res = emu_erk(method, P, y0, t_end, t_eval=te)
    st = res["state"][0]
    assert st["status"] == 0 and st["t"] == t_end and st["next_eval"] == len(te)
    assert st["nfev"] == sol.nfev, (st["nfev"], sol.nfev)
    assert st["n_rejected"] >= 1                                   # the controller's rejection branch is exercised
    want = np.moveaxis(sol.y.reshape(5, 200, -1), 2, 0)
    assert np.max(np.abs(res["snapshots"][0] - want)) <= STATE_GATE[method]
    assert np.max(np.abs(res["y"][0] - want[-1])) <= STATE_GATE[method]
    stages = 3 if method == "RK23" else 12
    dense = 0 if method == "RK23" else 3 * 4                       # DOP853: 4 steps sample a t_eval point
    assert st["nfev"] == 1 + stages * (st["n_accepted"] + st["n_rejected"]) + dense


@pytest.mark.parametrize("method", ["RK23", "DOP853"])
def test_explicit_kernel_events_and_dense_output_evaluations(emu_erk, method):
    """Events on the dense output: counts and root times as SciPy's.  DOP853 spends its three extra dense-output
    evaluations only in steps that SciPy asks for the dense output (a t_eval point or an event), so nfev matches SciPy
    with and without t_eval and events; monitoring never changes the trajectory."""
    pde, y0 = event_start()
    P = mb.derive_column_params(pde)
    t_end = 1.5e-4
    te = [0.3e-4, 1e-4]
    po = oracle.kernel_params(pde)
    plain = None
    for t_eval, events in (((), False), (te, False), ((), True), (te, True)):
        # (solve_ivp itself: oracle.integrate always passes a t_eval)
        sol = solve_ivp(oracle.rhs_fn(po), (0, t_end), y0[0].ravel(), method=method, first_step=1e-6, rtol=1e-3,
                        atol=1e-3, t_eval=list(t_eval) or None, events=oracle.event_fns(po, 200) if events else None)
        res = emu_erk(method, P, y0, t_end, t_eval=t_eval, events=events)
        assert res["state"]["nfev"][0] == sol.nfev, (t_eval, events, res["state"]["nfev"][0], sol.nfev)
        if plain is None:
            plain = res
        assert np.array_equal(res["y"], plain["y"])
        if events:
            want = [len(e) for e in sol.t_events]
            assert sum(want) >= 3 and list(res["event_counts"][0]) == want
            for k in range(7):
                assert np.max(np.abs(res["event_times"][0, k, :want[k]] - sol.t_events[k]), initial=0.0) <= 1e-12
        if len(t_eval):
            got = np.moveaxis(res["snapshots"][0], 0, 2).reshape(1000, -1)
            assert np.max(np.abs(got - sol.y)) <= STATE_GATE[method]


@pytest.mark.parametrize("method", ["RK23", "DOP853"])
def test_step_budget_and_resume_equal_a_whole_run_bit_for_bit(emu_erk, method):
    """Five columns of a lattice through the four warps of one CTA, cut into budgets of 7 attempts and resumed from the
    returned state: y, t, h_abs, step counts, t_eval samples and events equal the uninterrupted run bit for bit; nfev
    differs by exactly one evaluation of f(y) per resume."""
    pde, y0 = event_start()
    lat = mb.sweep_lattice(pde, 1, 1, 5)
    P = mb.derive_column_params(lat)
    Y = np.repeat(y0, 5, 0)
    t_end = 1e-4
    te = [0.0, 0.4e-4, t_end]
    whole = emu_erk(method, P, Y, t_end, t_eval=te, events=True)
    assert np.all(whole["state"]["status"] == 0)
    r = emu_erk(method, P, Y, t_end, t_eval=te, events=True, max_steps=7)
    resumes = np.zeros(5, np.int64)
    while np.any(r["state"]["status"] == 1):
        resumes += r["state"]["status"] == 1
        nxt = emu_erk(method, P, r["y"], t_end, t_eval=te, events=True, max_steps=7, state=r["state"],
                      counts=r["event_counts"], times=r["event_times"])
        keep = np.isnan(nxt["snapshots"])
        nxt["snapshots"][keep] = r["snapshots"][keep]
        r = nxt
    assert resumes.min() >= 2
    assert np.array_equal(r["y"], whole["y"])
    for k in ("t", "h_abs", "n_accepted", "n_rejected", "status", "next_eval"):
        assert np.array_equal(r["state"][k], whole["state"][k]), k
    assert np.array_equal(r["state"]["nfev"] - whole["state"]["nfev"], resumes)
    assert np.array_equal(r["snapshots"], whole["snapshots"], equal_nan=True)
    assert np.array_equal(r["event_counts"], whole["event_counts"]) and whole["event_counts"].sum() >= 5
    assert np.array_equal(r["event_times"], whole["event_times"], equal_nan=True)
    one = {k: (float(v[4]) if np.ndim(v) else v) for k, v in lat.items()}
    s4 = oracle.integrate(one, method=method, t_span=(0, t_end), t_eval=te, events=True, y0=y0[0].ravel(),
                          first_step=1e-6)
    assert whole["state"]["nfev"][4] == s4.nfev
    assert list(whole["event_counts"][4]) == [len(e) for e in s4.t_events]


@pytest.mark.parametrize("method", ["RK23", "DOP853"])
def test_time_varying_dPhi_and_ragged_grid_under_emulation(emu_erk, method):
    """The VD instantiation (MARLPDE_FLAG_VAR_DPHI): a flagged column follows SciPy on the oracle's model variant, a plain
    column of the same launch is bit-identical to the default instantiation; and an odd grid of 33 cells."""
    base = oracle.default_scenario() | SCEN_A
    var = base | {"time_varying_dPhi": True}
    P = np.concatenate([mb.derive_column_params(var), mb.derive_column_params(base)])
    Y = np.repeat(mb.initial_state(base), 2, 0)
    sol = oracle.integrate(var, method=method, t_span=(0, 1e-4), t_eval=[1e-4], events=False, first_step=1e-6)
    res = emu_erk(method, P, Y, 1e-4, t_eval=[1e-4], flags=_cabi.FLAG_VAR_DPHI)
    ref = emu_erk(method, P[1:], Y[1:], 1e-4, t_eval=[1e-4])
    assert np.all(res["state"]["status"] == 0) and res["state"]["nfev"][0] == sol.nfev
    assert np.max(np.abs(res["y"][0] - sol.y.reshape(5, 200))) <= STATE_GATE[method]
    assert np.array_equal(res["y"][1], ref["y"][0])
    pde = base | {"N": 33}
    sol = oracle.integrate(pde, method=method, t_span=(0, 5e-3), t_eval=[5e-3], events=False, first_step=1e-5)
    res = emu_erk(method, mb.derive_column_params(pde), mb.initial_state(pde), 5e-3, t_eval=[5e-3], first_step=1e-5)
    assert res["state"]["nfev"][0] == sol.nfev
    assert np.max(np.abs(res["y"][0] - sol.y.reshape(5, 33))) <= STATE_GATE[method]
