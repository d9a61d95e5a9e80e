"""Forward sensitivities of the BDF integrator on the GPU (marlpde_bdf_sens_integrate[_dev], bdf_kernel<., ., true>):
the state's path is bit-identical to the kernel without sensitivities, s = dy/d eps agrees with central differences of
the device integration at tight tolerance, does not depend on the batch order, agrees with the emulated kernel, and the
sweep driver stores it."""
import os
from dataclasses import asdict

import numpy as np
import pytest

import lheureux_oracle as oracle
import marlpde_b200 as mb

pytestmark = pytest.mark.gpu
np.seterr(all="ignore")
SCEN_A = {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}


def _S_direction(pde):
    S, D0Ca = pde["sedimentationrate"], pde["D0Ca"]
    return {"sedimentationrate": 1.0, "Xstar": -D0Ca / S ** 2, "Tstar": -2.0 * D0Ca / S ** 3}


def _state_fields(r):
    y = r.y.cpu().numpy() if hasattr(r.y, "cpu") else np.asarray(r.y)
    snaps = r.snapshots.cpu().numpy() if hasattr(r.snapshots, "cpu") else np.asarray(r.snapshots)
    return dict(y=y, snaps=snaps, state=r.state.tobytes(), nlu=r.nlu, njev=r.njev, it=r.newton_iterations,
                fail=r.newton_failures, ec=r.event_counts, et=r.event_times)


def _assert_same_path(a, b):
    fa, fb = _state_fields(a), _state_fields(b)
    for k in fa:
        if isinstance(fa[k], bytes):
            assert fa[k] == fb[k], k
        else:
            assert np.array_equal(fa[k], fb[k], equal_nan=True), k


@pytest.fixture(scope="module")
def lattice64():
    lat = mb.sweep_lattice(oracle.default_scenario(), 4, 4, 4)
    sd = mb.sensitivity_directions(lat, ["k2", "DCO3", _S_direction(lat)])
    return lat, sd


@pytest.mark.parametrize("path", ["host", "device"])
def test_state_path_is_bit_identical_with_sensitivities(lattice64, path):
    """64 lattice columns to t = 0.05 with events and t_eval, P = 3, through the host-pointer and the device path."""
    import torch
    lat, sd = lattice64
    P, y0 = mb.derive_column_params(lat), mb.initial_state(lat)
    if path == "device":
        y0 = torch.from_numpy(y0).cuda()
    kw = dict(t_span=(0, 0.05), first_step=1e-6, t_eval=[0.0, 0.02, 0.05], events=True, event_capacity=16)
    a = mb.integrate_bdf_batch(y0, P, **kw)
    b = mb.integrate_bdf_batch(y0, P, sensitivities=sd, **kw)
    _assert_same_path(a, b)
    s = b.sens_y.cpu().numpy() if path == "device" else b.sens_y
    assert s.shape == (64, 3, 5, 200) and np.all(np.isfinite(s[b.status == 0]))
    assert np.all(b.sens_stats[:, 0] > 0)
    ss = b.sensitivities.cpu().numpy() if path == "device" else b.sensitivities
    assert np.array_equal(ss[:, :, 0], sd.w)


def test_sensitivities_match_central_differences_on_the_device():
    """At rtol = atol = 1e-9, s(T) along k2, b, DCO3, PhiIni and the consistent S direction matches the central difference
    of the device integration itself (step 1e-3 pbar) to 1e-4 of max |s| — scenario A, N = 200, to t = 0.004."""
    pde = oracle.default_scenario() | SCEN_A
    dirs = ["k2", "b", "DCO3", "PhiIni", _S_direction(pde)]
    sd = mb.sensitivity_directions(pde, dirs)
    kw = dict(t_span=(0, 0.004), first_step=1e-7, rtol=1e-9, atol=1e-9)
    r = mb.integrate_bdf_batch(mb.initial_state(pde), mb.derive_column_params(pde), sensitivities=sd, **kw)
    assert r.status[0] == 0 and r.sens_stats[0, 2] == 0
    for k, d in enumerate(dirs):
        coef = {d: 1.0} if isinstance(d, str) else d
        pbar = min(abs(pde[q]) / abs(c) for q, c in coef.items() if pde[q] != 0 and c != 0)
        h = 1e-3 * pbar
        ys = []
        for sgn in (1.0, -1.0):
            q = dict(pde)
            for key, c in coef.items():
                q[key] = pde[key] + sgn * h * c
            ys.append(mb.integrate_bdf_batch(mb.initial_state(q), mb.derive_column_params(q), **kw).y[0])
        fd = (ys[0] - ys[1]) / (2 * h)
        err = np.max(np.abs(r.sens_y[0, k] - fd)) / np.max(np.abs(r.sens_y[0, k]))
        assert err <= 1e-4, (sd.names[k], err)


def test_batch_order_independence(lattice64):
    """A column's s does not depend on where it sits in the batch (bit for bit)."""
    lat, sd = lattice64
    P, y0 = mb.derive_column_params(lat), mb.initial_state(lat)
    perm = np.random.default_rng(3).permutation(64)
    kw = dict(t_span=(0, 0.02), first_step=1e-6, t_eval=[0.01, 0.02])
    a = mb.integrate_bdf_batch(y0, P, sensitivities=sd, **kw)
    sp = mb.SensitivityDirections(names=sd.names, params_pm=np.ascontiguousarray(sd.params_pm[perm]),
                                  inv2sigma=np.ascontiguousarray(sd.inv2sigma[perm]), w=np.ascontiguousarray(sd.w[perm]),
                                  pbar=np.ascontiguousarray(sd.pbar[perm]))
    b = mb.integrate_bdf_batch(np.ascontiguousarray(y0[perm]), np.ascontiguousarray(P[perm]), sensitivities=sp, **kw)
    assert np.array_equal(a.sens_y[perm], b.sens_y)
    assert np.array_equal(a.sensitivities[perm], b.sensitivities, equal_nan=True)
    assert np.array_equal(a.sens_stats[perm], b.sens_stats)


def test_device_agrees_with_the_emulated_kernel():
    """One column (scenario A, 33 cells, to t = 0.0275 with events) on the device and under the SIMT emulator: same step
    counts, and s within 1e-8 of max |s| (the host build's libm and fma contraction differ from the device's)."""
    import test_emu_sensitivity as emu_tests
    run = emu_tests.emu._fixture_function() if hasattr(emu_tests.emu, "_fixture_function") else emu_tests.emu.__wrapped__()
    pde = oracle.default_scenario() | SCEN_A | {"N": 33}
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    sd = mb.sensitivity_directions(pde, ["k2", "PhiIni"])
    e = run(P, y0, 0.0275, t_eval=[0.0275], events=True, first_step=5e-7, sens=sd)
    d = mb.integrate_bdf_batch(y0, P, t_span=(0, 0.0275), first_step=5e-7, t_eval=[0.0275], events=True,
                               event_capacity=16, sensitivities=sd)
    assert d.n_accepted[0] == e["state"]["n_accepted"][0] and d.nlu[0] == e["stats"][0, 1]
    for k in range(2):
        err = np.max(np.abs(d.sens_y[0, k] - e["sens_y"][0, k])) / np.max(np.abs(e["sens_y"][0, k]))
        assert err <= 1e-8, (sd.names[k], err)


def test_sweep_driver_stores_sensitivities(tmp_path):
    """integrate_equations_batch(..., sensitivities=[...]) with method BDF writes the dataset `sensitivities`
    (B, P, 5, N, n_t) and the direction names; hdf5lite reads them back.  Other methods refuse."""
    from marlpde.Evolve_scenario import integrate_equations_batch
    from marlpde.parameters import Map_Scenario, Solver, Tracker
    from marlpde_b200 import hdf5lite
    sweep = mb.sweep_lattice(asdict(Map_Scenario()) | SCEN_A, 2, 2, 1)
    tr = asdict(Tracker()) | {"t_eval": np.array([0.0, 0.01])}
    out = str(tmp_path / "sweep")
    r = integrate_equations_batch(asdict(Solver(method="BDF")) | {"t_span": (0, 0.01)}, tr, sweep, store_folder=out,
                                  sensitivities=["k2", "DCO3"])
    assert np.all(r.status == 0)
    with hdf5lite.File(os.path.join(out, "LMAHeureuxPorosityDiff_sweep.hdf5"), "r") as f:
        s = np.asarray(f["sensitivities"][...])
        assert s.shape == (4, 2, 5, 200, 2)
        assert np.array_equal(s, np.transpose(r.sensitivities, (0, 1, 3, 4, 2)), equal_nan=True)
        assert f.attrs["sensitivity_directions"].split("\n") == ["k2", "DCO3"]
    with pytest.raises(NotImplementedError):
        integrate_equations_batch(asdict(Solver(method="Radau")) | {"t_span": (0, 0.01)}, tr, sweep,
                                  sensitivities=["k2"])
