"""The batched explicit Runge-Kutta kernel (csrc/erk_batch.cu) on the B200: RK23 and DOP853 against live SciPy
(`solve_ivp(method="RK23" | "DOP853")` on the oracle RHS), with the gates of the RK45 tests (test_gpu_rk45.py).

One gate is looser for DOP853: t_eval samples INSIDE a step are compared at 5e-8 instead of 1e-9.  DOP853's error
estimate cancels about five orders of magnitude on this RHS, so the summation order of K^T E5 (the kernel's fma chain
against SciPy's BLAS dgemv) moves each step size in its 10th digit; at the stability limit where the explicit methods
run here, the seventh-order interpolant of a step is sensitive to that.  Measured under emulation (identical
arithmetic) at t = 0.002: 1.3e-8 in scenario A, 4.6e-10 / 1.6e-11 in the other two cases, while end states agree to
7e-11 and nfev is identical (tests/test_emu_explicit.py)."""
import os
from dataclasses import asdict

import numpy as np
import pytest
from numpy.testing import assert_allclose

import lheureux_oracle as oracle
import marlpde_b200 as mb

pytestmark = pytest.mark.gpu
np.seterr(all="ignore")

METHODS = ["RK23", "DOP853"]
STAGES = {"RK23": 3, "DOP853": 12}
NFEV_SLACK = {"RK23": 6, "DOP853": 27}                 # two attempts (and one dense output for DOP853)
SAMPLE_GATE = {"RK23": 1e-9, "DOP853": 5e-8}
SCEN_A = {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}


def run(method, *a, **kw):
    return {"RK23": mb.integrate_rk23_batch, "DOP853": mb.integrate_dop853_batch}[method](*a, **kw)


def _case(cases, name):
    c = cases[name]
    return oracle.default_scenario() | c["overrides"], c["first_step"]


def _dense_steps(res, method):
    """Steps that evaluated DOP853's extra dense-output stages, from the nfev identity."""
    extra = res.nfev - 1 - STAGES[method] * res.n_attempts
    assert np.all(extra % 3 == 0) and np.all(extra >= 0)
    return extra // 3 if method == "DOP853" else extra


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("name", ["scenario_A", "high_porosity", "matlab"])
def test_three_scenarios_short_horizon_against_scipy(stepper_golden, name, method):
    _, cases = stepper_golden
    pde, fs = _case(cases, name)
    te = [0.0, 0.0007, 0.0013, 0.002]
    sol = oracle.integrate(pde, method=method, t_span=(0, 0.002), t_eval=te, events=False, first_step=fs)
    res = run(method, mb.initial_state(pde), mb.derive_column_params(pde), t_span=(0, 0.002), first_step=fs, t_eval=te)
    assert res.status[0] == 0 and res.t[0] == 0.002 and res.next_eval[0] == 4
    assert abs(int(res.nfev[0]) - sol.nfev) <= NFEV_SLACK[method], (int(res.nfev[0]), sol.nfev)
    want = sol.y.reshape(5, 200, -1)
    got = res.solutions(0)
    assert np.max(np.abs(got[:, :, -1] - want[:, :, -1])) <= 1e-9
    assert np.max(np.abs(got - want)) <= SAMPLE_GATE[method]
    # nfev identities: RK23 1 + 3 attempts; DOP853 1 + 12 attempts + 3 per step that sampled t_eval (4 steps here)
    assert int(_dense_steps(res, method)[0]) == (0 if method == "RK23" else 4)


@pytest.mark.parametrize("method", METHODS)
def test_events_default_scenario_match_scipy(method):
    """Default Map_Scenario to t = 0.03: porosity crosses 1 once (event 4) and max W changes sign 11 times (event 6) —
    the same counts as SciPy's, root times to 1e-7; monitoring does not change the trajectory."""
    pde = oracle.default_scenario()
    sol = oracle.integrate(pde, method=method, t_span=(0, 0.03), t_eval=[0, 0.03], events=True)
    res = run(method, mb.initial_state(pde), mb.derive_column_params(pde), t_span=(0, 0.03), first_step=1e-6,
              t_eval=[0, 0.03], events=True, event_capacity=32)
    assert res.status[0] == 0
    assert [len(e) for e in sol.t_events] == list(res.event_counts[0]) == [0, 0, 0, 0, 1, 0, 11]
    cap = res.event_times.shape[2]
    for k in range(7):
        got = np.sort(res.event_times[0, k, :min(int(res.event_counts[0, k]), cap)])
        assert_allclose(got, sol.t_events[k], rtol=0, atol=1e-7)
    plain = run(method, mb.initial_state(pde), mb.derive_column_params(pde), t_span=(0, 0.03), first_step=1e-6,
                t_eval=[0, 0.03])
    assert np.array_equal(plain.y, res.y) and np.array_equal(plain.n_attempts, res.n_attempts)
    dense_ev = _dense_steps(res, method)[0]
    dense_plain = _dense_steps(plain, method)[0]
    if method == "DOP853":                           # 2 sampling steps + the steps that located events
        assert dense_plain == 2 and 2 < dense_ev <= 2 + 12
    assert abs(int(res.nfev[0]) - sol.nfev) <= 60


@pytest.mark.parametrize("method", METHODS)
def test_columns_independent_of_batch_order_and_device_path(method):
    import torch
    lat = mb.sweep_lattice(oracle.default_scenario() | SCEN_A, 2, 2, 2)
    P, y0 = mb.derive_column_params(lat), mb.initial_state(lat)
    te = [0.0, 0.001, 0.002]
    host = run(method, y0, P, t_span=(0, 0.002), t_eval=te, events=True, event_capacity=8)
    perm = np.random.default_rng(3).permutation(8)
    shuf = run(method, y0[perm], P[perm], t_span=(0, 0.002), t_eval=te, events=True, event_capacity=8)
    assert np.array_equal(shuf.y, host.y[perm]) and np.array_equal(shuf.nfev, host.nfev[perm])
    assert np.array_equal(shuf.snapshots, host.snapshots[perm], equal_nan=True)
    dev = run(method, torch.from_numpy(y0).cuda(), P, t_span=(0, 0.002), t_eval=te, events=True, event_capacity=8)
    assert np.array_equal(dev.y.cpu().numpy(), host.y)
    assert np.array_equal(dev.snapshots.cpu().numpy(), host.snapshots)
    assert np.array_equal(dev.nfev, host.nfev) and np.array_equal(dev.event_counts, host.event_counts)


@pytest.mark.parametrize("method", METHODS)
def test_step_budget_and_resume_is_bit_identical(method):
    pde = oracle.default_scenario() | SCEN_A
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    whole = run(method, y0, P, t_span=(0, 0.002), t_eval=[0.001, 0.002])
    r = run(method, y0, P, t_span=(0, 0.002), t_eval=[0.001, 0.002], max_steps=100)
    hops, snaps = 0, np.array(r.snapshots)
    while r.status[0] == 1:
        assert r.t[0] < 0.002
        r = run(method, r.y, P, t_span=(0, 0.002), t_eval=[0.001, 0.002], max_steps=100, state=r.state)
        keep = np.isnan(snaps)
        snaps[keep] = np.asarray(r.snapshots)[keep]
        hops += 1
    assert hops >= 3 and r.status[0] == 0
    assert np.array_equal(r.y, whole.y) and np.array_equal(snaps, whole.snapshots)
    assert r.h_abs[0] == whole.h_abs[0] and r.n_accepted[0] == whole.n_accepted[0]
    assert r.nfev[0] == whole.nfev[0] + hops


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("n_cells,ncol", [(33, 3), (257, 2), (2000, 1)])
def test_ragged_shapes_and_large_grids(method, n_cells, ncol):
    pde = oracle.default_scenario() | SCEN_A | {"N": n_cells}
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    t_end = 2e-4 * (200 / n_cells) ** 2 if n_cells > 200 else 2e-4
    fs = 1e-6 * min(1.0, (200 / n_cells) ** 2)
    res = run(method, np.repeat(y0, ncol, 0), np.repeat(P, ncol), t_span=(0, t_end), first_step=fs, t_eval=[0, t_end])
    sol = oracle.integrate(pde, method=method, t_span=(0, t_end), t_eval=[0, t_end], events=False, first_step=fs)
    assert np.all(res.status == 0) and np.all(res.t == t_end)
    assert np.all(np.abs(res.nfev - sol.nfev) <= NFEV_SLACK[method]), (res.nfev, sol.nfev)
    for c in range(ncol):
        assert np.max(np.abs(res.solutions(c)[:, :, -1] - sol.y[:, -1].reshape(5, n_cells))) <= 1e-9


@pytest.mark.parametrize("method", METHODS)
def test_time_varying_dPhi_against_scipy(method):
    base = oracle.default_scenario() | SCEN_A
    var = base | {"time_varying_dPhi": True}
    P = np.concatenate([mb.derive_column_params(var), mb.derive_column_params(base)])
    y0 = np.repeat(mb.initial_state(base), 2, 0)
    sol = oracle.integrate(var, method=method, t_span=(0, 0.002), t_eval=[0, 0.002], events=False)
    res = run(method, y0, P, t_span=(0, 0.002), t_eval=[0, 0.002])
    plain = run(method, y0[1:], P[1:], t_span=(0, 0.002), t_eval=[0, 0.002])
    assert np.all(res.status == 0) and abs(int(res.nfev[0]) - sol.nfev) <= NFEV_SLACK[method]
    assert np.max(np.abs(res.solutions(0)[:, :, -1] - sol.y[:, -1].reshape(5, 200))) <= 1e-9
    assert np.array_equal(res.y[1], plain.y[0])


@pytest.mark.parametrize("method", METHODS)
def test_full_Tstar_against_reference_fixtures(stepper_golden, fixtures_reference, method):
    """The three reference regression cases to T* in one launch, at the reference's tolerances (test_regression.py:
    rtol 0.1, atol 0.01; the Matlab cross-check atol 0.05 on cells 2..)."""
    _, cases = stepper_golden
    names = ["scenario_A", "high_porosity", "matlab"]
    pdes = [_case(cases, n) for n in names]
    P = np.concatenate([mb.derive_column_params(p) for p, _ in pdes])
    y0 = np.concatenate([mb.initial_state(p) for p, _ in pdes])
    res = run(method, y0, P, t_span=(0, 1), first_step=np.array([fs for _, fs in pdes]), t_eval=[0.0, 1.0])
    assert np.all(res.status == 0) and np.all(res.t == 1.0)
    for c, name in enumerate(names):
        got = res.solutions(c)[:, :, -1]
        if name != "matlab":
            assert_allclose(got, fixtures_reference[name][-1], rtol=0.1, atol=0.01)
        else:
            m = fixtures_reference["matlab"]
            x, _ = oracle.grid_coords(pdes[c][0])
            interp = np.stack([np.interp(x * pdes[c][0]["Xstar"], np.linspace(0, 500, 201), m[f, :, 0]) for f in range(5)])
            assert_allclose(got[:, 2:], interp[:, 2:], atol=0.05)


@pytest.fixture()
def in_tmp_cwd(tmp_path, monkeypatch):
    work = tmp_path / "run"
    work.mkdir()
    monkeypatch.chdir(work)
    return tmp_path


@pytest.mark.parametrize("method", METHODS)
def test_drop_in_runs_on_the_device_and_matches_the_scipy_stepper(in_tmp_cwd, monkeypatch, method):
    """integrate_equations(Solver(method=...)) steps on the device; MARLPDE_SCIPY_STEPPER=1 keeps SciPy's stepper over
    the CUDA RHS.  The two agree to 1e-9 at t = 0.002; the batch entry point and the sweep accept the method."""
    import time
    import marlpde_b200
    from marlpde.Evolve_scenario import integrate_equations, integrate_equations_batch
    from marlpde.parameters import Map_Scenario, Solver, Tracker
    scen = asdict(Map_Scenario()) | SCEN_A
    short = {"t_span": (0, 0.002)}
    tr = asdict(Tracker()) | {"t_eval": np.array([0.0, 0.002])}
    calls = []
    real = getattr(marlpde_b200, f"integrate_{method.lower()}_batch")
    monkeypatch.setattr(marlpde_b200, f"integrate_{method.lower()}_batch", lambda *a, **k: calls.append(1) or real(*a, **k))
    a, covered, _, _, _ = integrate_equations(asdict(Solver(method=method)) | short, dict(tr), dict(scen))
    assert calls == [1] and covered == pytest.approx(scen["Tstar"] * 0.002)
    monkeypatch.setenv("MARLPDE_SCIPY_STEPPER", "1")
    time.sleep(1.1)            # the output folder is a one-second timestamp, like upstream
    b, _, _, _, _ = integrate_equations(asdict(Solver(method=method)) | short, dict(tr), dict(scen))
    assert calls == [1]
    assert_allclose(a, b, rtol=0, atol=1e-9)
    monkeypatch.delenv("MARLPDE_SCIPY_STEPPER")
    sweep = mb.sweep_lattice(scen, 1, 2, 2)
    tr2 = asdict(Tracker()) | {"t_eval": np.array([0.0, 0.002])}
    r = integrate_equations_batch(asdict(Solver(method=method)) | short, tr2, sweep, store_folder=str(in_tmp_cwd / "sw"))
    assert np.all(r.status == 0) and os.path.exists(in_tmp_cwd / "sw" / "LMAHeureuxPorosityDiff_sweep.hdf5")
    s = mb.sweep.sweep_rk45(sweep, t_span=(0, 0.002), t_eval=[0.0, 0.002], method=method)
    assert np.all(s.status == 0)
    assert np.array_equal(s.y, np.asarray(r.y)) and np.array_equal(s.nfev, r.nfev)
