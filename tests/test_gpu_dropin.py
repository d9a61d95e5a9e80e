"""The reference's own regression tests (tests/Regression_test/test_regression.py:21-148), run through
the drop-in mirror: same imports, same calls, same tolerances — `integrate_equations` with the default
`Solver()` (Radau, rtol = atol = 1e-3), final-time fields against the reference's HDF5 fixtures (decoded
once into tests/golden/fixtures_reference.npz; h5py is not installed here) — plus the HDF5 output layout
(Evolve_scenario.py:157-178) and the RK45 / SciPy-stepper routes of the same entry point, the SciPy Radau stepper
driving the CUDA RHS to T* included."""
import glob
import os
from dataclasses import asdict

import numpy as np
import pytest
from numpy.testing import assert_allclose

from marlpde.parameters import Map_Scenario, Solver, Tracker
from marlpde.Evolve_scenario import integrate_equations, integrate_equations_batch
from marlpde_b200 import hdf5lite
from marlpde_b200.pde_standin import CartesianGrid, ScalarField

pytestmark = pytest.mark.gpu
np.seterr(all="ignore")


@pytest.fixture()
def in_tmp_cwd(tmp_path, monkeypatch):
    """integrate_equations writes ../Results/<timestamp>/ relative to the CWD (Evolve_scenario.py:157-159)."""
    work = tmp_path / "run"
    work.mkdir()
    monkeypatch.chdir(work)
    return tmp_path


def test_integration_Scenario_A(fixtures_reference, in_tmp_cwd):
    rtol, atol = 0.1, 0.01
    Scenario_parameters = asdict(Map_Scenario()) | {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    solver = asdict(Solver())
    assert solver["method"] == "Radau"
    last_field_sol, covered_time, depths, Xstar, store_folder = integrate_equations(solver, asdict(Tracker()),
                                                                                    Scenario_parameters)
    assert_allclose(last_field_sol, fixtures_reference["scenario_A"][-1], rtol=rtol, atol=atol)
    assert "backend" not in solver                                   # mutated like upstream (:102)
    assert covered_time == Scenario_parameters["Tstar"] and Xstar == Scenario_parameters["Xstar"]
    # ---- output file: same datasets, shapes and root attributes as upstream (:170-178)
    files = glob.glob(str(in_tmp_cwd / "Results" / "*" / "LMAHeureuxPorosityDiff.hdf5"))
    assert len(files) == 1 and os.path.samefile(os.path.dirname(files[0]), store_folder)
    with hdf5lite.File(files[0], "r") as f:
        assert sorted(f.keys()) == sorted(["solutions", "times"] + [f"event_{k}" for k in range(7)])
        assert f["solutions"].shape == (5, 200, 2) and np.array_equal(f["times"][:], [0.0, 1.0])
        assert np.array_equal(f["solutions"][:, :, -1], last_field_sol)
        assert f.attrs["method"] == "Radau" and f.attrs["N"] == 200 and f.attrs["Phi0"] == 0.6
        assert "jac_sparsity" not in f.attrs and "backend" not in f.attrs
        # scenario A: CA decays to numerical zero (1e-17) in the dissolution zone after t ~ 0.06, so the sign
        # changes of min(y) = min(CA) (events 0, 1) are round-off: SciPy itself reports 0.2488 at rtol 1e-3 and
        # 0.2939 at 1e-8.  What is pinned: both monitors see the same crossings, no other monitor fires.
        assert f["event_0"].shape[0] >= 1 and np.array_equal(f["event_0"][:], f["event_1"][:])
        assert all(f[f"event_{k}"].shape == (0,) for k in (2, 3, 4, 5, 6))


def test_high_porosity_integration(fixtures_reference, in_tmp_cwd):
    rtol, atol = 0.1, 0.01
    Scenario_parameters = asdict(Map_Scenario()) | {"Phi0": 0.8, "PhiIni": 0.8, "PhiNR": 0.8}
    Solver_parms = asdict(Solver()) | {"first_step": 5e-7}
    last_field_sol, _, _, _, _ = integrate_equations(Solver_parms, asdict(Tracker()), Scenario_parameters)
    assert_allclose(last_field_sol, fixtures_reference["high_porosity"][-1], rtol=rtol, atol=atol)


def test_cross_check_with_Matlab_output(fixtures_reference, in_tmp_cwd):
    atol = 0.05
    Matlab_output = fixtures_reference["matlab"]
    Matlab_depths = np.linspace(0, 500, Matlab_output.shape[1])
    Scenario_parameters = asdict(Map_Scenario()) | {"Phi0": 0.5, "PhiIni": 0.5, "PhiNR": 0.5, "k3": 0.01, "k4": 0.01}
    Xstar, max_depth = Scenario_parameters["Xstar"], Scenario_parameters["max_depth"]
    last_field_sol, _, _, _, _ = integrate_equations(asdict(Solver()), asdict(Tracker()), Scenario_parameters)
    Number_of_depths = Scenario_parameters["N"]
    Python_depth_grid = CartesianGrid([[0, max_depth / Xstar]], [Number_of_depths], periodic=False)
    Python_plotting_depths = ScalarField.from_expression(Python_depth_grid, "x").data * Xstar
    Matlab_output_interpolated = np.empty((Matlab_output.shape[0], Number_of_depths))
    for field in range(Matlab_output.shape[0]):
        Matlab_output_interpolated[field, :] = np.interp(Python_plotting_depths, Matlab_depths, Matlab_output[field, :, 0])
    assert_allclose(last_field_sol[:, 2:], Matlab_output_interpolated[:, 2:], atol=atol)


def test_rk45_and_scipy_stepper_routes(fixtures_reference, in_tmp_cwd, monkeypatch):
    """Same entry point, other `method`s: RK45 runs on the persistent kernel; with MARLPDE_SCIPY_STEPPER=1
    SciPy steps and the GPU only evaluates the RHS (the reference's own loop, Evolve_scenario.py:104-109)."""
    scen = asdict(Map_Scenario()) | {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    short = {"t_span": (0, 0.002)}
    tr = asdict(Tracker()) | {"t_eval": np.array([0.0, 0.002])}
    import time
    a, covered, _, _, _ = integrate_equations(asdict(Solver(method="RK45")) | short, dict(tr), dict(scen))
    monkeypatch.setenv("MARLPDE_SCIPY_STEPPER", "1")
    time.sleep(1.1)            # the output folder is a one-second timestamp, like upstream (:157-159)
    b, _, _, _, _ = integrate_equations(asdict(Solver(method="RK45")) | short, dict(tr), dict(scen))
    time.sleep(1.1)
    assert_allclose(a, b, rtol=0, atol=1e-9)
    assert covered == pytest.approx(scen["Tstar"] * 0.002)
    c, _, _, _, _ = integrate_equations(asdict(Solver(method="LSODA")) | short, dict(tr), dict(scen))
    assert_allclose(a, c, rtol=0, atol=2e-2)              # LSODA with the reference's lband = uband = 1


def test_scipy_radau_stepper_with_cuda_rhs_matches_fixture(fixtures_reference, in_tmp_cwd, monkeypatch):
    """The reference's own loop to T* (Evolve_scenario.py:104-109): SciPy's Radau with the reference's jac_sparsity
    (finite-difference Jacobian by column groups) steps scenario A, every RHS evaluation is the CUDA kernel through
    `eq.fun_numba`; final fields against the reference's fixture at its tolerances."""
    import marlpde_b200

    def no_device_stepper(*a, **kw):
        raise AssertionError("MARLPDE_SCIPY_STEPPER=1 must leave the stepping to SciPy")
    monkeypatch.setattr(marlpde_b200, "integrate_radau_batch", no_device_stepper)
    monkeypatch.setenv("MARLPDE_SCIPY_STEPPER", "1")
    scen = asdict(Map_Scenario()) | {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
    solver = asdict(Solver())
    assert solver["method"] == "Radau" and solver["jac_sparsity"] is not None
    last_field_sol, covered_time, _, _, _ = integrate_equations(solver, asdict(Tracker()), scen)
    assert_allclose(last_field_sol, fixtures_reference["scenario_A"][-1], rtol=0.1, atol=0.01)
    assert covered_time == scen["Tstar"]


@pytest.mark.parametrize("n_cells", [16, 1000])
def test_rk45_drop_in_outside_the_on_chip_grid_range(in_tmp_cwd, n_cells):
    """integrate_equations(method="RK45") monitors the 7 events at any N like the reference (Evolve_scenario.py:104-109):
    grids below 32 or above 640 cells run on the streaming kernels, events included."""
    import lheureux_oracle as oracle
    scale = min(1.0, (200 / n_cells) ** 2)
    t_end = 300 * 2.6e-6 * scale
    scen = asdict(Map_Scenario()) | {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6, "N": n_cells}
    solver = asdict(Solver(method="RK45")) | {"t_span": (0, t_end), "first_step": 1e-6 * scale}
    tr = asdict(Tracker()) | {"t_eval": np.array([0.0, t_end])}
    last, covered, depths, xstar, folder = integrate_equations(solver, tr, dict(scen))
    assert last.shape == (5, n_cells) and covered == pytest.approx(scen["Tstar"] * t_end)
    sol = oracle.integrate(scen, method="RK45", t_span=(0, t_end), t_eval=[0, t_end], events=True, first_step=1e-6 * scale)
    assert_allclose(last, sol.y[:, -1].reshape(5, n_cells), rtol=0, atol=1e-9)
    with hdf5lite.File(os.path.join(folder, "LMAHeureuxPorosityDiff.hdf5"), "r") as f:
        assert f["solutions"].shape == (5, n_cells, 2)
        for k in range(7):
            assert np.asarray(f[f"event_{k}"]).shape == (len(sol.t_events[k]),)


def test_batch_entry_point_radau_and_rk45(in_tmp_cwd):
    import marlpde_b200 as mb
    sweep = mb.sweep_lattice(asdict(Map_Scenario()) | {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}, 2, 2, 2)
    tr = asdict(Tracker()) | {"t_eval": np.array([0.0, 0.01])}
    out = str(in_tmp_cwd / "sweep")
    r = integrate_equations_batch(asdict(Solver()) | {"t_span": (0, 0.01)}, tr, sweep, store_folder=out)
    e = integrate_equations_batch(asdict(Solver(method="RK45")) | {"t_span": (0, 0.01)}, tr, sweep)
    assert np.all(r.status == 0) and np.all(e.status == 0)
    assert np.max(np.abs(np.asarray(r.y) - np.asarray(e.y))) <= 6e-2           # implicit vs explicit at rtol 1e-3, in the initial transient
    with hdf5lite.File(os.path.join(out, "LMAHeureuxPorosityDiff_sweep.hdf5"), "r") as f:
        assert f["solutions"].shape == (8, 5, 200, 2) and f["status"].shape == (8,)
