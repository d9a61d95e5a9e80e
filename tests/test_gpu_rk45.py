"""GPU parity of the persistent RK45 kernel (marlpde_rk45_integrate through the C ABI) against
SciPy's RK45 on the CPU oracle — the reference's own stepper (Evolve_scenario.py:104-109).

Tolerances: the solver runs at rtol=atol=1e-3; two correct implementations of the same step
sequence differ only by round-off (FMA, summation order), which the survey measured at <=1e-9 on
the end state with identical nfev.  Gates: short horizon <=1e-9 abs with |nfev difference| <= 12
(two step attempts), full T* <=1e-5 abs vs SciPy and the reference's regression tolerances
(rtol=0.1, atol=0.01) vs its fixtures."""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import lheureux_oracle as oracle
import marlpde_b200 as mb

pytestmark = pytest.mark.gpu
np.seterr(all="ignore")


def _case(cases, name):
    c = cases[name]
    return oracle.default_scenario() | c["overrides"], c["first_step"]


@pytest.mark.parametrize("name", ["scenario_A", "high_porosity", "matlab"])
def test_short_horizon_matches_scipy_golden(stepper_golden, name):
    g, cases = stepper_golden
    pde, fs = _case(cases, name)
    key = f"{name}/RK45/t0.002/tol0.001"
    te = g[key + "/t"]
    res = mb.integrate_rk45_batch(mb.initial_state(pde), mb.derive_column_params(pde), t_span=(0, 0.002),
                                  first_step=fs, rtol=1e-3, atol=1e-3, t_eval=te)
    assert res.status[0] == 0 and res.t[0] == 0.002 and res.next_eval[0] == te.size
    assert abs(int(res.nfev[0]) - int(g[key + "/counts"][0])) <= 12
    assert res.nfev[0] == 1 + 6 * (res.n_accepted[0] + res.n_rejected[0])
    ref = g[key + "/y"].reshape(5, 200, -1)
    assert_allclose(res.solutions(0), ref, rtol=0, atol=1e-9)        # all 5 dense-output samples
    assert np.array_equal(res.solutions(0)[:, :, 0], mb.initial_state(pde)[0])   # t_eval[0] = t0 -> y0
    assert_allclose(res.y[0], ref[:, :, -1], rtol=0, atol=1e-9)


def test_live_scipy_on_lattice_columns_with_dense_output():
    """Columns with different parameters share one CTA; each must match its own SciPy run."""
    base = oracle.default_scenario() | {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    pde = mb.sweep_lattice(base, 2, 2, 2)
    te = np.array([0.0, 1e-5, 3.3e-4, 7e-4, 1e-3])
    res = mb.integrate_rk45_batch(mb.initial_state(pde), mb.derive_column_params(pde), t_span=(0, 1e-3),
                                  first_step=1e-6, t_eval=te)
    assert np.all(res.status == 0)
    for c in (0, 3, 5, 7):
        one = {k: (v[c] if np.ndim(v) else v) for k, v in pde.items()}
        sol = oracle.integrate(one, method="RK45", t_span=(0, 1e-3), t_eval=te, events=False)
        assert abs(int(res.nfev[c]) - sol.nfev) <= 12, c
        assert_allclose(res.solutions(c), sol.y.reshape(5, 200, -1), rtol=0, atol=1e-9)


def test_columns_are_independent_and_deterministic():
    """A column's trajectory must not depend on which other columns share its CTA or on queue order."""
    base = oracle.default_scenario()
    pde = mb.sweep_lattice(base, 3, 3, 3)
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    full = mb.integrate_rk45_batch(y0, P, t_span=(0, 5e-4), first_step=5e-7)
    again = mb.integrate_rk45_batch(y0, P, t_span=(0, 5e-4), first_step=5e-7)
    assert np.array_equal(full.y, again.y) and np.array_equal(full.nfev, again.nfev)
    for c in (0, 13, 26):
        alone = mb.integrate_rk45_batch(y0[c:c + 1], P[c:c + 1], t_span=(0, 5e-4), first_step=5e-7)
        assert np.array_equal(alone.y[0], full.y[c]) and alone.nfev[0] == full.nfev[c]
    rev = mb.integrate_rk45_batch(y0[::-1].copy(), P[::-1].copy(), t_span=(0, 5e-4), first_step=5e-7)
    assert np.array_equal(rev.y[::-1], full.y)


def test_warp_order_does_not_change_results(monkeypatch):
    """The kernel deals its physical warps out to the column ranges in an order chosen for scheduler balance
    (rk45_persistent.cu: sPerm).  Which warp integrates which cells must not matter: the automatic order, the
    identity and an arbitrary permutation give bit-identical trajectories, counters and event times."""
    pde = mb.sweep_lattice(oracle.default_scenario(), 2, 2, 2)
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    kw = dict(t_span=(0, 5e-4), first_step=5e-7, t_eval=[2.5e-4, 5e-4], events=True, event_capacity=16)
    auto = mb.integrate_rk45_batch(y0, P, **kw)
    for order in ("identity", "9,8,7,6,5,4,3,2,1,0", "0,1,4,3,2,5,6,7,8,9"):
        monkeypatch.setenv("MARLPDE_RK45_WARP_PERM", order)
        res = mb.integrate_rk45_batch(y0, P, **kw)
        assert np.array_equal(res.y, auto.y) and np.array_equal(res.snapshots, auto.snapshots), order
        assert np.array_equal(res.nfev, auto.nfev) and np.array_equal(res.event_counts, auto.event_counts), order
        assert np.array_equal(res.event_times, auto.event_times, equal_nan=True), order


def test_step_budget_and_resume_is_bit_identical():
    pde = oracle.default_scenario() | {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    te = np.linspace(0, 1e-3, 4)
    whole = mb.integrate_rk45_batch(y0, P, t_span=(0, 1e-3), t_eval=te)
    part = mb.integrate_rk45_batch(y0, P, t_span=(0, 1e-3), t_eval=te, max_steps=100)
    assert part.status[0] == 1 and 0 < part.t[0] < 1e-3
    hops = 1
    while part.status[0] == 1:
        snaps = part.snapshots
        part = mb.integrate_rk45_batch(part.y, P, t_span=(0, 1e-3), t_eval=te, max_steps=100, state=part.state)
        keep = np.isnan(part.snapshots)
        part.snapshots[keep] = snaps[keep]
        hops += 1
    assert hops >= 3 and part.status[0] == 0
    assert part.n_accepted[0] == whole.n_accepted[0] and part.n_rejected[0] == whole.n_rejected[0]
    assert np.array_equal(part.y, whole.y)
    assert np.array_equal(part.snapshots, whole.snapshots)


def test_ragged_shapes_and_many_columns():
    """N not a multiple of 32, one and two columns per CTA, more columns than resident slots."""
    for n_cells, ncol in ((33, 5), (100, 9), (257, 3), (608, 2)):
        pde = oracle.default_scenario() | {"N": n_cells, "Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
        P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
        t_end = 2e-4 * (200 / n_cells) ** 2 if n_cells > 200 else 2e-4
        res = mb.integrate_rk45_batch(np.repeat(y0, ncol, 0), np.repeat(P, ncol), t_span=(0, t_end),
                                      first_step=1e-6 * min(1.0, (200 / n_cells) ** 2), t_eval=[0, t_end])
        sol = oracle.integrate(pde, method="RK45", t_span=(0, t_end), t_eval=[0, t_end], events=False,
                               first_step=1e-6 * min(1.0, (200 / n_cells) ** 2))
        assert np.all(res.status == 0), n_cells
        assert np.all(np.abs(res.nfev - sol.nfev) <= 12), (n_cells, res.nfev, sol.nfev)
        for c in range(ncol):
            assert_allclose(res.solutions(c)[:, :, -1], sol.y[:, -1].reshape(5, n_cells), rtol=0, atol=1e-9)
    big = mb.sweep_lattice(oracle.default_scenario(), 10, 10, 10)              # 1000 columns > 444 slots
    res = mb.integrate_rk45_batch(mb.initial_state(big), mb.derive_column_params(big), t_span=(0, 2e-5),
                                  first_step=5e-7)
    assert np.all(res.status == 0) and np.all(res.t == 2e-5) and np.all(np.isfinite(res.y))


def test_unsupported_and_degenerate_inputs():
    from marlpde_b200._cabi import MarlpdeError
    pde = oracle.default_scenario()
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    with pytest.raises(MarlpdeError, match="n_cells"):         # the smallest grid has two cells
        mb.integrate_rk45_batch(np.full((1, 5, 1), 0.5), P)
    res = mb.integrate_rk45_batch(y0[:0], P[:0])
    assert res.y.shape == (0, 5, 200)
    # a state that is already non-finite collapses the step size like SciPy: status -1, never hangs
    bad = y0.copy()
    bad[0, 4, 10] = np.nan
    res = mb.integrate_rk45_batch(bad, P, t_span=(0, 1e-3))
    assert res.status[0] == -1 and res.n_accepted[0] == 0


def test_device_tensor_path_matches_host_path():
    import torch
    pde = mb.sweep_lattice(oracle.default_scenario(), 2, 2, 2)
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    te = [0.0, 1e-4, 2e-4]
    host = mb.integrate_rk45_batch(y0, P, t_span=(0, 2e-4), first_step=5e-7, t_eval=te)
    dev = mb.integrate_rk45_batch(torch.from_numpy(y0).cuda(), P, t_span=(0, 2e-4), first_step=5e-7, t_eval=te)
    assert np.array_equal(dev.y.cpu().numpy(), host.y)
    assert np.array_equal(dev.snapshots.cpu().numpy(), host.snapshots)
    assert np.array_equal(dev.nfev, host.nfev)


@pytest.mark.parametrize("name,fixture", [("scenario_A", "scenario_A"), ("high_porosity", "high_porosity"),
                                          ("matlab", None)])
def test_full_Tstar_against_scipy_rk45_and_reference_fixtures(stepper_golden, fixtures_reference, name, fixture):
    """BASELINE.json configs[0]: N=200, RK45 to the full T*.  SciPy needs 90-160 s per column for
    this (committed golden, tests/golden/make_stepper_golden.py); the GPU runs it live."""
    g, cases = stepper_golden
    pde, fs = _case(cases, name)
    key = f"{name}/RK45/t1/tol0.001"
    res = mb.integrate_rk45_batch(mb.initial_state(pde), mb.derive_column_params(pde), t_span=(0, 1),
                                  first_step=fs, rtol=1e-3, atol=1e-3, t_eval=[0.0, 1.0])
    ref = g[key + "/y"].reshape(5, 200, -1)[:, :, -1]
    ref_nfev = int(g[key + "/counts"][0])
    assert res.status[0] == 0 and res.t[0] == 1.0
    got = res.solutions(0)[:, :, -1]
    if name != "matlab":
        assert abs(int(res.nfev[0]) - ref_nfev) <= 1e-4 * ref_nfev  # same step sequence up to round-off
        assert_allclose(got, ref, rtol=0, atol=1e-5)
    else:
        # The Matlab case is round-off chaotic in its cCO3 top boundary layer: two SciPy runs whose
        # first_step differs by 1e-9 relative end 1.3e-2 apart in cell 0 (decaying ~1.7x per cell) and
        # 354 RHS calls apart (committed golden).  The GPU must sit inside that CPU-vs-CPU envelope.
        pert = g[key + "/y_end_first_step_times_1p000000001"]
        noise_nfev = abs(int(g[key + "/nfev_first_step_times_1p000000001"]) - ref_nfev)
        assert abs(int(res.nfev[0]) - ref_nfev) <= 10 * noise_nfev
        d = np.abs(got - ref)
        assert d[[0, 1, 4]].max() <= 1e-5 and d[2].max() <= 2e-4
        envelope = 4 * np.abs(pert[3] - ref[3]).max() * 1.6 ** -np.arange(200.0) + 1e-5
        assert np.all(d[3] <= envelope), (d[3][:16], envelope[:16])
    if fixture is not None:                                          # test_regression.py:29-30, :52-53
        assert_allclose(got, fixtures_reference[fixture][-1], rtol=0.1, atol=0.01)
    else:                                                            # test_regression.py:103, :136-148
        m = fixtures_reference["matlab"]
        x, _ = oracle.grid_coords(pde)
        interp = np.stack([np.interp(x * pde["Xstar"], np.linspace(0, 500, 201), m[f, :, 0]) for f in range(5)])
        assert_allclose(got[:, 2:], interp[:, 2:], atol=0.05)


# ---- event monitors (LHeureux_model.py:524-593; ivp.py find_active_events / brentq) -----------------
def _event_lists(res, column):
    cap = res.event_times.shape[2]
    return [np.sort(res.event_times[column, k, :min(int(res.event_counts[column, k]), cap)]) for k in range(7)]


def test_events_default_scenario_match_scipy():
    """Default Map_Scenario to t = 0.03: porosity crosses 1 once (event 4) and max W changes sign
    seven times (event 6).  Same counts as SciPy, root times to 1e-7 (the two trajectories agree to
    ~1e-9, the roots are located to 4 eps on either side)."""
    pde = oracle.default_scenario()
    sol = oracle.integrate(pde, method="RK45", t_span=(0, 0.03), t_eval=[0, 0.03], events=True)
    res = mb.integrate_rk45_batch(mb.initial_state(pde), mb.derive_column_params(pde), t_span=(0, 0.03),
                                  first_step=1e-6, t_eval=[0, 0.03], events=True, event_capacity=32)
    assert res.status[0] == 0 and abs(int(res.nfev[0]) - sol.nfev) <= 60
    assert [len(e) for e in sol.t_events] == list(res.event_counts[0]) == [0, 0, 0, 0, 1, 0, 7]
    for got, want in zip(_event_lists(res, 0), sol.t_events):
        assert_allclose(got, want, rtol=0, atol=1e-7)
    assert_allclose(res.solutions(0)[:, :, -1], sol.y[:, -1].reshape(5, 200), rtol=0, atol=1e-7)
    # monitoring must not change the trajectory
    plain = mb.integrate_rk45_batch(mb.initial_state(pde), mb.derive_column_params(pde), t_span=(0, 0.03),
                                    first_step=1e-6, t_eval=[0, 0.03])
    assert np.array_equal(plain.y, res.y) and np.array_equal(plain.nfev, res.nfev)


def test_events_synthetic_state_six_monitors_and_capacity():
    """A state that starts outside the physical bounds (CA<0, CC<0, CA+CC>1, Phi>1 in single cells)
    re-enters them within t = 4e-3: monitors 0-4 and 6 fire; columns sharing a CTA keep their own
    event lists; a small capacity truncates the stored times but not the counts."""
    pde = oracle.default_scenario() | {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    y0 = mb.initial_state(pde)
    y0[0, 0, 50] = -2e-3
    y0[0, 1, 60] = -1e-3
    y0[0, 0, 100] = 0.705
    y0[0, 4, 150] = 1.0005
    sol = oracle.integrate(pde, method="RK45", t_span=(0, 4e-3), t_eval=[0, 4e-3], events=True, y0=y0[0])
    want_counts = [len(e) for e in sol.t_events]
    assert want_counts == [1, 1, 1, 1, 2, 0, 2]
    P = mb.derive_column_params(pde)
    Y = np.concatenate([y0, mb.initial_state(pde), y0, y0])          # columns 0, 2, 3 perturbed, 1 plain
    res = mb.integrate_rk45_batch(Y, np.repeat(P, 4), t_span=(0, 4e-3), first_step=1e-6, t_eval=[0, 4e-3],
                                  events=True, event_capacity=8)
    assert np.all(res.status == 0)
    for c in (0, 2, 3):
        assert list(res.event_counts[c]) == want_counts
        for got, want in zip(_event_lists(res, c), sol.t_events):
            assert_allclose(got, want, rtol=0, atol=1e-9)
    assert np.all(res.event_counts[1] == 0)
    assert np.array_equal(res.y[0], res.y[2]) and np.array_equal(res.event_times[0], res.event_times[3], equal_nan=True)
    small = mb.integrate_rk45_batch(y0, P, t_span=(0, 4e-3), first_step=1e-6, events=True, event_capacity=1)
    assert list(small.event_counts[0]) == want_counts and small.event_times.shape == (1, 7, 1)
    assert small.event_times[0, 4, 0] == res.event_times[0, 4, 0]


def test_events_survive_resume():
    """Stopping on a step budget and resuming gives the same event lists as one uninterrupted run."""
    pde = oracle.default_scenario()
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    whole = mb.integrate_rk45_batch(y0, P, t_span=(0, 0.029), first_step=1e-6, events=True, event_capacity=16)
    part = mb.integrate_rk45_batch(y0, P, t_span=(0, 0.029), first_step=1e-6, events=True, event_capacity=16,
                                   max_steps=7000)
    times = [list(e) for e in _event_lists(part, 0)]
    while part.status[0] == 1:
        part = mb.integrate_rk45_batch(part.y, P, t_span=(0, 0.029), events=True, event_capacity=16,
                                       max_steps=7000, state=part.state)
        for k, e in enumerate(_event_lists(part, 0)):
            times[k] += list(e)
    assert part.status[0] == 0 and np.array_equal(part.y, whole.y)
    for k in range(7):
        assert np.array_equal(np.asarray(times[k]), _event_lists(whole, 0)[k])


# ---- depth grids that do not fit on chip: the streaming path (csrc/rk45_streaming.cu) ---------------
@pytest.mark.parametrize("window", ["auto", "large"])
@pytest.mark.parametrize("n_cells,ncol", [(2000, 3), (5000, 1), (641, 2), (16, 2), (1257, 2)])
def test_streaming_path_matches_scipy(n_cells, ncol, window, monkeypatch):
    """BASELINE.json configs[3] (SURVEY.md §8d config 4): fixed budget of ~2000 steps, t_end and
    first_step scaled with (200/N)^2 (the explicit step is stability bound), state at t_end against SciPy
    RK45 on the oracle.  Same stepper semantics as the on-chip kernel: nfev within two attempts.
    window: the launcher's choice (256-cell windows for every batch here) or the 640-cell windows forced."""
    if window == "large":
        monkeypatch.setenv("MARLPDE_RK45_TILE", "large")
    else:
        monkeypatch.delenv("MARLPDE_RK45_TILE", raising=False)
    pde = oracle.default_scenario() | {"N": n_cells, "Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    scale = min(1.0, (200 / n_cells) ** 2)
    t_end, fs = 600 * 2.6e-6 * scale, 1e-6 * scale
    te = [0.0, 0.4 * t_end, t_end]
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    res = mb.integrate_rk45_batch(np.repeat(y0, ncol, 0), np.repeat(P, ncol), t_span=(0, t_end), first_step=fs, t_eval=te)
    sol = oracle.integrate(pde, method="RK45", t_span=(0, t_end), t_eval=te, events=False, first_step=fs)
    assert np.all(res.status == 0) and np.all(res.t == t_end) and np.all(res.next_eval == 3)
    assert np.all(np.abs(res.nfev - sol.nfev) <= 12), (res.nfev, sol.nfev)
    want = sol.y.reshape(5, n_cells, -1)
    for c in range(ncol):
        assert_allclose(res.solutions(c), want, rtol=0, atol=1e-9)
        assert_allclose(res.y[c], want[:, :, -1], rtol=0, atol=1e-9)
    assert np.array_equal(res.y[0], res.y[-1])


def test_streaming_window_sizes_agree(monkeypatch):
    """The tile kernel's two window sizes: 640-cell windows (large batches) and 256-cell windows (small batches, chosen by
    the launcher when the large ones would leave more than half of the SMs idle).  The window size only changes the order
    in which the per-window error sums are added."""
    n_cells = 2000
    pde = oracle.default_scenario() | {"N": n_cells, "Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    P, y0 = np.repeat(mb.derive_column_params(pde), 3), np.repeat(mb.initial_state(pde), 3, 0)
    t_end, fs = 300 * 2.6e-6 / 100, 1e-6 / 100
    run = lambda: mb.integrate_rk45_batch(y0, P, t_span=(0, t_end), first_step=fs, t_eval=[0.5 * t_end, t_end])
    monkeypatch.setenv("MARLPDE_RK45_TILE", "large")
    large = run()
    monkeypatch.setenv("MARLPDE_RK45_TILE", "small")
    small = run()
    monkeypatch.delenv("MARLPDE_RK45_TILE")
    auto = run()
    assert np.all(large.status == 0) and large.n_attempts[0] >= 200
    assert np.array_equal(auto.y, small.y)                       # 3 columns x 4 large windows: the launcher picks small ones
    assert np.array_equal(small.nfev, large.nfev) and np.max(np.abs(small.y - large.y)) <= 1e-12
    assert np.max(np.abs(small.snapshots - large.snapshots)) <= 1e-12


def test_streaming_path_resume_device_tensors_and_budget():
    import torch
    n_cells = 1000
    pde = oracle.default_scenario() | {"N": n_cells, "Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    t_end, fs = 700 * 2.6e-6 / 25, 1e-6 / 25
    whole = mb.integrate_rk45_batch(y0, P, t_span=(0, t_end), first_step=fs, t_eval=[0, t_end])
    assert whole.status[0] == 0
    part = mb.integrate_rk45_batch(y0, P, t_span=(0, t_end), first_step=fs, max_steps=300)
    assert part.status[0] in (1, 2) and part.n_attempts[0] == 300 and 0 < part.t[0] < t_end
    rest = mb.integrate_rk45_batch(part.y, P, t_span=(0, t_end), state=part.state)
    assert rest.status[0] == 0 and rest.n_attempts[0] == whole.n_attempts[0]
    assert_allclose(rest.y, whole.y, rtol=0, atol=1e-12)             # K1 is re-evaluated on resume: same bits expected
    dev = mb.integrate_rk45_batch(torch.from_numpy(y0).cuda(), P, t_span=(0, t_end), first_step=fs, t_eval=[0, t_end])
    assert np.array_equal(dev.y.cpu().numpy(), whole.y) and np.array_equal(dev.snapshots.cpu().numpy(), whole.snapshots)


def test_host_path_scratch_pool_is_reused_and_released():
    """The host-pointer entry points take their device scratch from a stream-ordered pool that keeps blocks between
    calls (cudaMalloc/cudaFree cost up to 130 ms per call on the bench box); results do not depend on it, the pool can
    be trimmed, and the calling thread's current device is left alone."""
    from marlpde_b200 import _cabi
    pde = oracle.default_scenario()
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    _cabi.lib().marlpde_release_cached_memory()
    a = mb.integrate_rk45_batch(y0, P, t_span=(0, 1e-4), first_step=1e-6)
    b = mb.integrate_rk45_batch(y0, P, t_span=(0, 1e-4), first_step=1e-6)        # served from the pool
    assert np.array_equal(a.y, b.y) and np.array_equal(a.nfev, b.nfev)
    assert _cabi.lib().marlpde_release_cached_memory() >= 1          # number of per-device pools trimmed
    c = mb.integrate_rk45_batch(y0, P, t_span=(0, 1e-4), first_step=1e-6)
    assert np.array_equal(a.y, c.y)


def test_streaming_path_20000_cells_matches_scipy():
    """BASELINE.json configs[3] at its largest grid: N = 20 000, one column and a batch of 8, 600 step attempts from
    t = 0 against SciPy RK45 on the oracle (1.1 ms per RHS call on the CPU)."""
    n_cells = 20000
    pde = oracle.default_scenario() | {"N": n_cells, "Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    scale = (200 / n_cells) ** 2
    t_end, fs = 500 * 2.6e-6 * scale, 1e-6 * scale
    te = [0.0, 0.5 * t_end, t_end]
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    sol = oracle.integrate(pde, method="RK45", t_span=(0, t_end), t_eval=te, events=False, first_step=fs)
    want = sol.y.reshape(5, n_cells, -1)
    for ncol in (1, 8):
        res = mb.integrate_rk45_batch(np.repeat(y0, ncol, 0), np.repeat(P, ncol), t_span=(0, t_end), first_step=fs, t_eval=te)
        assert np.all(res.status == 0) and np.all(res.t == t_end) and np.all(res.next_eval == 3)
        assert np.all(np.abs(res.nfev - sol.nfev) <= 12), (res.nfev, sol.nfev)
        assert res.n_attempts[0] >= 400
        assert_allclose(res.solutions(0), want, rtol=0, atol=1e-9)
        assert np.array_equal(res.y[0], res.y[-1])


@pytest.mark.parametrize("n_cells", [1000, 1257, 16])
def test_streaming_path_events_match_scipy(n_cells):
    """The 7 monitors on depth grids outside the on-chip range (the reference monitors at any N,
    LHeureux_model.py:524-593, Evolve_scenario.py:107-109): a state that starts outside the physical bounds in single
    cells re-enters them, so monitors 0-4 and 6 fire; counts equal SciPy's, root times to 1e-9 (scaled grid: the
    explicit step is stability bound, t_end ~ (200/N)^2).  A column without excursions in the same batch stays silent,
    and monitoring does not change the trajectory."""
    pde = oracle.default_scenario() | {"N": n_cells, "Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    scale = min(1.0, (200 / n_cells) ** 2)
    t_end, fs = 1500 * 2.6e-6 * scale, 1e-6 * scale
    y0 = mb.initial_state(pde)
    pick = lambda frac: min(n_cells - 1, int(frac * n_cells))
    y0[0, 0, pick(0.25)] = -2e-3 * scale
    y0[0, 1, pick(0.30)] = -1e-3 * scale
    y0[0, 0, pick(0.50)] = 0.7 + 5e-3 * scale
    y0[0, 4, pick(0.75)] = 1.0 + 5e-4 * scale
    sol = oracle.integrate(pde, method="RK45", t_span=(0, t_end), t_eval=[0, t_end], events=True, y0=y0[0], first_step=fs)
    want_counts = [len(e) for e in sol.t_events]
    assert sum(c > 0 for c in want_counts) >= 4, want_counts
    P = mb.derive_column_params(pde)
    Y = np.concatenate([y0, mb.initial_state(pde), y0])
    res = mb.integrate_rk45_batch(Y, np.repeat(P, 3), t_span=(0, t_end), first_step=fs, t_eval=[0, t_end],
                                  events=True, event_capacity=8)
    assert np.all(res.status == 0) and np.all(np.abs(res.nfev[[0, 2]] - sol.nfev) <= 12)
    for c in (0, 2):
        assert list(res.event_counts[c]) == want_counts
        for got, want in zip(_event_lists(res, c), sol.t_events):
            assert_allclose(got, want, rtol=0, atol=1e-9 * max(scale, 1e-3))
    assert np.all(res.event_counts[1] == 0)
    assert np.array_equal(res.event_times[0], res.event_times[2], equal_nan=True)
    plain = mb.integrate_rk45_batch(Y, np.repeat(P, 3), t_span=(0, t_end), first_step=fs, t_eval=[0, t_end])
    assert np.array_equal(plain.y, res.y) and np.array_equal(plain.nfev, res.nfev)
    assert np.array_equal(plain.snapshots, res.snapshots)
    # device-tensor route and a run cut into batches (events located in one batch are not located again in the next)
    import torch
    dev = mb.integrate_rk45_batch(torch.from_numpy(Y).cuda(), np.repeat(P, 3), t_span=(0, t_end), first_step=fs,
                                  t_eval=[0, t_end], events=True, event_capacity=8)
    assert np.array_equal(dev.event_counts, res.event_counts) and np.array_equal(dev.event_times, res.event_times, equal_nan=True)
    per_call = max(4, int(res.n_attempts.max()) // 4)
    part = mb.integrate_rk45_batch(Y, np.repeat(P, 3), t_span=(0, t_end), first_step=fs, events=True, event_capacity=8,
                                   max_steps=per_call)
    counts = part.event_counts.copy()
    hops = 1
    while np.any(part.status >= 1):
        part = mb.integrate_rk45_batch(part.y, np.repeat(P, 3), t_span=(0, t_end), events=True, event_capacity=8,
                                       max_steps=per_call, state=part.state)
        counts += part.event_counts
        hops += 1
    assert hops >= 3 and np.array_equal(counts, res.event_counts) and np.array_equal(part.y, res.y)


@pytest.mark.parametrize("n_cells", [200, 1000])
def test_time_varying_dPhi_model_variant_matches_scipy(n_cells):
    """SURVEY 8(f) row 4: the per-cell porosity diffusion coefficient dPhi = auxcon F Phi^3 / (1 - Phi)
    (LHeureux_model.py:222-223, :430-431) as a kernel template flag, on-chip (N = 200) and streaming (N = 1000) kernels,
    against SciPy RK45 on the oracle variant; flagged and plain columns share one launch and the plain ones are
    bit-identical to a launch without any flagged column."""
    base = oracle.default_scenario() | {"N": n_cells, "Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    var = base | {"time_varying_dPhi": True}
    scale = min(1.0, (200 / n_cells) ** 2)
    t_end, fs = 400 * 2.6e-6 * scale, 1e-6 * scale
    P = np.concatenate([mb.derive_column_params(var), mb.derive_column_params(base), mb.derive_column_params(var)])
    assert list(P["model_flags"]) == [1, 0, 1] and P["auxcon"][0] > 0
    Y = np.repeat(mb.initial_state(base), 3, 0)
    res = mb.integrate_rk45_batch(Y, P, t_span=(0, t_end), first_step=fs, t_eval=[0, t_end], events=True, event_capacity=4)
    plain = mb.integrate_rk45_batch(Y[:1], P[1:2], t_span=(0, t_end), first_step=fs, t_eval=[0, t_end], events=True,
                                    event_capacity=4)
    assert np.all(res.status == 0)
    assert np.array_equal(res.y[1], plain.y[0]) and res.nfev[1] == plain.nfev[0]
    assert np.array_equal(res.y[0], res.y[2])
    sol = oracle.integrate(var, method="RK45", t_span=(0, t_end), t_eval=[0, t_end], events=False, first_step=fs)
    assert abs(int(res.nfev[0]) - sol.nfev) <= 12
    assert_allclose(res.y[0], sol.y[:, -1].reshape(5, n_cells), rtol=0, atol=1e-9)
    assert np.max(np.abs(res.y[0][4] - res.y[1][4])) > 1e-7          # a different model, visibly


def test_async_host_entry_point_overlaps_and_matches_sync():
    """marlpde_rk45_integrate_async: copies, launch and scratch release enqueued on the caller's stream, no
    synchronisation inside; two batches on two streams give the results of the blocking call."""
    import ctypes as C
    import torch
    from marlpde_b200 import _cabi, batch
    pde = mb.sweep_lattice(oracle.default_scenario(), 2, 2, 4)
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    want = mb.integrate_rk45_batch(y0, P, t_span=(0, 2e-4), first_step=5e-7, events=True, event_capacity=4)
    lib = _cabi.lib()
    o = _cabi.RK45Options(t_bound=2e-4, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=0, n_eval=0,
                          event_capacity=4, flags=_cabi.FLAG_EVENTS, quantum=0)
    halves, streams = [], [torch.cuda.Stream(), torch.cuda.Stream()]
    for k, s in enumerate(streams):
        sl = slice(8 * k, 8 * k + 8)
        bufs = dict(y=torch.from_numpy(y0[sl].copy()).pin_memory(),
                    p=torch.from_numpy(P[sl].view(np.uint8).copy()).pin_memory(),
                    st=torch.from_numpy(batch.make_state(8, 0.0, 5e-7).view(np.uint8).copy()).pin_memory(),
                    ec=torch.zeros((8, 7), dtype=torch.int32).pin_memory(),
                    et=torch.full((8, 7, 4), float("nan"), dtype=torch.float64).pin_memory())
        _cabi.check(lib.marlpde_rk45_integrate_async(bufs["y"].data_ptr(), bufs["p"].data_ptr(), bufs["st"].data_ptr(), 8, 200,
                                                     C.byref(o), None, None, bufs["ec"].data_ptr(), bufs["et"].data_ptr(),
                                                     torch.cuda.current_device(), s.cuda_stream))
        halves.append(bufs)
    for s in streams:
        s.synchronize()
    got_y = np.concatenate([h["y"].numpy() for h in halves])
    got_ec = np.concatenate([h["ec"].numpy() for h in halves])
    assert np.array_equal(got_y, want.y) and np.array_equal(got_ec, want.event_counts)
    st = np.concatenate([h["st"].numpy().view(_cabi.STATE_DTYPE) for h in halves])
    assert np.array_equal(st["nfev"], want.nfev) and np.all(st["status"] == 0)
