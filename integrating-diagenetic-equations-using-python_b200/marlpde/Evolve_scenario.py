#!/usr/bin/env python
"""Scenario driver with the reference's interface (marlpde/Evolve_scenario.py):

    integrate_equations(solver_parms, tracker_parms, pde_parms)
        -> (last_fields (5, N), covered_time, depths, Xstar, store_folder)

and the same HDF5 output (`solutions` (5, N, n_t), `times`, `event_0..6`, parameters as root
attributes) under ../Results/<timestamp>/, but the time stepping runs on the B200:

  method == "RK45"   the persistent sm_100a kernel integrates the column on-chip
                     (csrc/rk45_persistent.cu), SciPy RK45 semantics incl. t_eval dense output and events;
  method == "Radau"  (the reference's default, parameters.py:213) the batched implicit kernel
                     (csrc/radau_batch.cu): SciPy Radau semantics, block-tridiagonal Newton solve;
  method == "BDF"    the batched variable-order BDF kernel (csrc/bdf_batch.cu): SciPy's BDF step for step on the
                     same block-tridiagonal solver;
  method == "LSODA"  SciPy's solve_ivp (ODEPACK's Fortran stepper, exactly what upstream runs) drives `eq.fun_numba`,
                     whose RHS is the CUDA kernel (one column per call); MARLPDE_LSODA_DEVICE=1 runs the column on
                     the device BDF kernel instead — LSODA leaves its Adams mode after ~25 steps on this stiff system
                     and is a variable-order BDF code from then on (csrc/bdf_batch.cu), `lband` / `uband` are then
                     ignored like `jac_sparsity`: the kernel's block-tridiagonal Jacobian is the exact structure;
  method == "RK23"   the batched explicit Runge-Kutta kernel (csrc/erk_batch.cu), SciPy RK23 step for step: same
  method == "DOP853" step control and error norm, the method's own dense output for t_eval and events (DOP853's
                     three extra stages only in steps that need them, as SciPy);
  MARLPDE_SCIPY_STEPPER=1 keeps SciPy's own stepper for every method, the RHS still evaluated by the CUDA kernel (one
                     column per call) — same arguments upstream passes (:104-109).

`integrate_equations_batch` is the sweep entry point: many parameter sets in one launch.
"""
from __future__ import annotations

import inspect
import os
import time
from dataclasses import asdict
from datetime import datetime
from types import SimpleNamespace

import numpy as np

import marlpde_b200 as _mb
from marlpde_b200 import hdf5lite
from marlpde_b200.pde_standin import CartesianGrid, ScalarField
from LHeureux_model import LMAHeureuxPorosityDiff
from parameters import Map_Scenario, Solver, Tracker

_EVENT_TEXT = ("any field at any depth crossed zero", "CA at any depth crossed zero",
               "CC at any depth crossed zero", "CA + CC at any depth crossed one",
               "the porosity at any depth crossed one", "U at any depth crossed zero",
               "W at any depth crossed zero")
_MESSAGES = {0: "The solver successfully reached the end of the integration interval.",
             -1: "Required step size is less than spacing between numbers.",
             1: "Step budget exhausted before reaching the end of the integration interval."}


def _build_model(pde_parms):
    """Grid, dissolution-zone masks and model object (reference :40-68)."""
    n = pde_parms["N"]
    xstar = pde_parms["Xstar"]
    depths = CartesianGrid([[0, pde_parms["max_depth"] / xstar]], [n], periodic=False)
    not_too_shallow = ScalarField.from_expression(depths, f"heaviside(x-{pde_parms['ShallowLimit'] / xstar}, 0)")
    not_too_deep = ScalarField.from_expression(depths, f"heaviside({pde_parms['DeepLimit'] / xstar}-x, 0)")
    accepted = set(inspect.signature(LMAHeureuxPorosityDiff).parameters)
    model_args = {k: v for k, v in pde_parms.items() if k in accepted}
    slices = [slice(i * n, (i + 1) * n) for i in range(5)]
    eq = LMAHeureuxPorosityDiff(depths, slices, not_too_shallow, not_too_deep, **model_args)
    state = eq.get_state(*(ScalarField(depths, pde_parms[k])
                           for k in ("CAIni", "CCIni", "cCaIni", "cCO3Ini", "PhiIni")))
    return depths, eq, state.data.ravel()


def _gpu_rk45(eq, y0, solver_parms, t_eval, n_cells, integrate=None):
    """One column through the persistent kernel (or `integrate`: the explicit RK23 / DOP853 kernel, same arguments and
    result type); returns an OdeResult look-alike."""
    known = {"first_step", "atol", "rtol", "t_span", "method", "dense_output", "max_step"}
    extra = set(solver_parms) - known
    if extra:
        raise TypeError(f"options not supported by the GPU {solver_parms.get('method', 'RK45')} path: {sorted(extra)}")
    integrate = integrate or _mb.integrate_rk45_batch
    # `dense_output=True` (parameters.py:221 has False) makes solve_ivp attach a callable OdeSolution as `sol.sol`;
    # upstream's driver never reads it (Evolve_scenario.py:104-183 uses sol.y, sol.t, sol.t_events only), so the flag is
    # accepted and stored with the other parameters; intermediate states come from `t_eval`, which IS the dense output
    # (quartic / cubic interpolant of the step, as SciPy) evaluated on the device.
    te = np.asarray(t_eval, dtype=np.float64) if t_eval is not None else np.array(solver_parms["t_span"], float)
    res = integrate(y0.reshape(1, 5, n_cells), eq.column_params, t_span=solver_parms["t_span"],
                    first_step=solver_parms.get("first_step", 1e-6),
                    rtol=solver_parms.get("rtol", 1e-3), atol=solver_parms.get("atol", 1e-6),
                    max_step=solver_parms.get("max_step", np.inf), t_eval=te,
                    events=True, event_capacity=4096)
    k = int(res.next_eval[0])
    status = int(res.status[0])
    t_events = [np.sort(res.event_times[0, e, :min(int(res.event_counts[0, e]), res.event_times.shape[2])])
                for e in range(7)]
    return SimpleNamespace(t=te[:k], y=res.solutions(0).reshape(5 * n_cells, k), t_events=t_events,
                           nfev=int(res.nfev[0]), njev=0, nlu=0, status=status, success=status >= 0,
                           message=_MESSAGES.get(status, "unknown status"), t_reached=float(res.t[0]))


def _gpu_implicit(eq, y0, solver_parms, t_eval, n_cells, kind="radau"):
    """One column through a batched implicit integrator — csrc/radau_batch.cu (SciPy Radau semantics) or
    csrc/bdf_batch.cu (SciPy BDF semantics) — with the block-tridiagonal Newton solve.  `jac_sparsity` (and LSODA's
    `lband` / `uband`) are accepted and ignored — the 5x5 block-tridiagonal structure is intrinsic to the kernels (it
    is the exact structure the reference's pattern approximates)."""
    known = {"first_step", "atol", "rtol", "t_span", "method", "dense_output", "max_step", "jac_sparsity", "lband", "uband"}
    extra = set(solver_parms) - known
    if extra:
        raise TypeError(f"options not supported by the GPU implicit path: {sorted(extra)}")
    integrate = _mb.integrate_radau_batch if kind == "radau" else _mb.integrate_bdf_batch
    # `dense_output=True` (parameters.py:221 has False) makes solve_ivp attach a callable OdeSolution as `sol.sol`;
    # upstream's driver never reads it (Evolve_scenario.py:104-183 uses sol.y, sol.t, sol.t_events only), so the flag is
    # accepted and stored with the other parameters; intermediate states come from `t_eval`, which IS the dense output
    # (quartic / cubic interpolant of the step, as SciPy) evaluated on the device.
    te = np.asarray(t_eval, dtype=np.float64) if t_eval is not None else np.array(solver_parms["t_span"], float)
    res = integrate(y0.reshape(1, 5, n_cells), eq.column_params, t_span=solver_parms["t_span"],
                    first_step=solver_parms.get("first_step", 1e-6),
                    rtol=solver_parms.get("rtol", 1e-3), atol=solver_parms.get("atol", 1e-6),
                    max_step=solver_parms.get("max_step", np.inf), t_eval=te, events=True, event_capacity=4096)
    k = int(res.next_eval[0])
    status = int(res.status[0])
    t_events = [np.sort(res.event_times[0, e, :min(int(res.event_counts[0, e]), res.event_times.shape[2])])
                for e in range(7)]
    return SimpleNamespace(t=te[:k], y=res.solutions(0).reshape(5 * n_cells, k), t_events=t_events,
                           nfev=int(res.nfev[0]), njev=int(res.njev[0]), nlu=int(res.nlu[0]), status=status,
                           success=status >= 0, message=_MESSAGES.get(status, "unknown status"),
                           t_reached=float(res.t[0]))


def _store(store_folder, stored_parms, field_solutions, times, t_events):
    os.makedirs(store_folder)
    stored_results = store_folder + "LMAHeureuxPorosityDiff.hdf5"
    with hdf5lite.File(stored_results, "w") as stored:
        stored.create_dataset("solutions", data=field_solutions)
        stored.create_dataset("times", data=times)
        for event_index, te in enumerate(t_events):
            stored.create_dataset("event_" + str(event_index), data=np.asarray(te, dtype=np.float64))
        stored.attrs.update(stored_parms)
    return stored_results


def integrate_equations(solver_parms, tracker_parms, pde_parms):
    """Integrate one sediment column; same contract as the reference's function (:19-183)."""
    xstar, tstar = pde_parms["Xstar"], pde_parms["Tstar"]
    n_cells = pde_parms["N"]
    depths, eq, y0 = _build_model(pde_parms)

    no_progress_updates = tracker_parms["no_progress_updates"]
    t0, end_time = solver_parms["t_span"][0], solver_parms["t_span"][1]
    backend = solver_parms["backend"]          # "numpy" and "numba" share one CUDA RHS here
    del solver_parms["backend"]                # mutated on purpose, as upstream (:102)
    assert backend in ("numpy", "numba"), backend

    start_computing = time.time()
    progress = 0
    scipy_stepper = os.environ.get("MARLPDE_SCIPY_STEPPER", "0") == "1"    # SciPy steps, the GPU only evaluates the RHS
    explicit = {"RK45": _mb.integrate_rk45_batch, "RK23": _mb.integrate_rk23_batch, "DOP853": _mb.integrate_dop853_batch}
    if solver_parms["method"] in explicit and not scipy_stepper:
        gpu_parms = {k: v for k, v in solver_parms.items() if k not in ("jac_sparsity", "lband", "uband")}
        sol = _gpu_rk45(eq, y0, gpu_parms, tracker_parms["t_eval"], n_cells, explicit[solver_parms["method"]])
        progress = (sol.t_reached - t0) / (end_time - t0)
    elif solver_parms["method"] == "Radau" and not scipy_stepper:
        sol = _gpu_implicit(eq, y0, solver_parms, tracker_parms["t_eval"], n_cells, "radau")
        progress = (sol.t_reached - t0) / (end_time - t0)
    elif not scipy_stepper and (solver_parms["method"] == "BDF" or (
            solver_parms["method"] == "LSODA" and os.environ.get("MARLPDE_LSODA_DEVICE", "0") == "1")):
        sol = _gpu_implicit(eq, y0, solver_parms, tracker_parms["t_eval"], n_cells, "bdf")
        progress = (sol.t_reached - t0) / (end_time - t0)
    else:
        from scipy.integrate import solve_ivp
        try:
            from tqdm import tqdm
        except ImportError:                     # progress bar is cosmetic
            tqdm = None
        bar = tqdm(total=no_progress_updates) if tqdm else SimpleNamespace(update=lambda n: None, n=0, close=lambda: None)
        try:
            progress_bar_args = [bar, (end_time - t0) / no_progress_updates, t0]
            sol = solve_ivp(eq.fun if backend == "numpy" else eq.fun_numba, y0=y0, **solver_parms,
                            t_eval=tracker_parms["t_eval"],
                            events=[eq.zeros, eq.zeros_CA, eq.zeros_CC, eq.ones_CA_plus_CC, eq.ones_Phi,
                                    eq.zeros_U, eq.zeros_W], args=progress_bar_args)
            progress = bar.n / no_progress_updates
        finally:
            bar.close()
    end_computing = time.time()

    print()
    print(f"Number of rhs evaluations = {sol.nfev} \n")
    print(f"Number of Jacobian evaluations = {sol.njev} \n")
    print(f"Number of LU decompositions = {sol.nlu} \n")
    print(f"Status = {sol.status} \n")
    print(f"Success = {sol.success} \n")
    for text, times in zip(_EVENT_TEXT, sol.t_events):
        print(f"Times, in years, at which {text}: " + ", ".join("%.2f" % (tstar * te) for te in times))
        print()
    print(f"Message from solve_ivp = {sol.message} \n")
    print(f"Time taken for solve_ivp is {end_computing - start_computing:.2e}s. \n")

    covered_time = tstar * end_time if sol.status == 0 else progress * tstar * end_time

    store_folder = "../Results/" + datetime.now().strftime("%d_%m_%Y_%H_%M_%S" + "/")
    while os.path.exists(store_folder):        # upstream's names have a one-second resolution (:157-159) and it needs
        time.sleep(0.1)                        # >= 0.2 s per run; a column takes ~30 ms here, so two runs can collide
        store_folder = "../Results/" + datetime.now().strftime("%d_%m_%Y_%H_%M_%S" + "/")
    stored_parms = solver_parms | tracker_parms | pde_parms
    stored_parms.pop("jac_sparsity", None)     # not storable as HDF5 metadata
    field_solutions = sol.y.reshape(5, n_cells, sol.y.shape[-1])
    _store(store_folder, stored_parms, field_solutions, sol.t, sol.t_events)
    return field_solutions[:, :, -1], covered_time, depths, xstar, store_folder


def integrate_equations_batch(solver_parms, tracker_parms, pde_parms, store_folder=None, device=0, sensitivities=None):
    """Parameter sweep: `pde_parms` is a Map_Scenario dictionary whose values may be arrays of
    shape (B,) (see marlpde_b200.sweep_lattice) or a list of such dictionaries.  All columns are
    integrated in one launch of the kernel `method` selects (RK45: persistent on-chip kernel; RK23, DOP853: the batched
    explicit Runge-Kutta kernel; Radau, BDF / LSODA: the batched implicit kernels).  Returns the marlpde_b200.RK45Result / RadauResult;
    with `store_folder` one HDF5 file per sweep is written (datasets `solutions` (B,5,N,n_t),
    `times`, `status`, `nfev`, `n_accepted`, `n_rejected`, `next_eval`, `t_reached`, `event_counts`).

    `sensitivities` (methods BDF and LSODA only): a list of directions as for marlpde_b200.sensitivity_directions (each a
    key of `pde_parms` or a {key: coefficient} dict), or the object that function returns.  The result then carries the
    forward sensitivities dy/d eps at fixed nondimensional time (RadauResult.sensitivities / sens_y / sens_stats), and
    the sweep file gains the dataset `sensitivities` (B, P, 5, N, n_t) and the attribute `sensitivity_directions`
    (the direction names, one per line)."""
    if isinstance(pde_parms, (list, tuple)):
        keys = pde_parms[0].keys()
        pde_parms = {k: (np.array([p[k] for p in pde_parms]) if k != "N" else pde_parms[0]["N"]) for k in keys}
    solver_parms = dict(solver_parms)
    solver_parms.pop("backend", None)
    method = solver_parms.get("method", "RK45")
    if method not in ("RK45", "RK23", "DOP853", "Radau", "BDF", "LSODA"):
        raise NotImplementedError("the batched on-device integrators implement method='RK45', 'RK23', 'DOP853', 'Radau', "
                                  "'BDF' and 'LSODA' (the latter on the BDF kernel: LSODA's stiff mode)")
    if sensitivities is not None and method not in ("BDF", "LSODA"):
        raise NotImplementedError("forward sensitivities are implemented on the BDF kernel (methods 'BDF' and 'LSODA')")
    params = _mb.derive_column_params(pde_parms)
    y0 = _mb.initial_state(pde_parms)
    extra = {}
    if sensitivities is not None:
        if not isinstance(sensitivities, _mb.SensitivityDirections):
            sensitivities = _mb.sensitivity_directions(pde_parms, sensitivities)
        extra = {"sensitivities": sensitivities}
    integrate = {"RK45": _mb.integrate_rk45_batch, "RK23": _mb.integrate_rk23_batch, "DOP853": _mb.integrate_dop853_batch,
                 "Radau": _mb.integrate_radau_batch}.get(method, _mb.integrate_bdf_batch)
    res = integrate(y0, params, t_span=solver_parms.get("t_span", (0, 1)),
                    first_step=solver_parms.get("first_step", 1e-6),
                    rtol=solver_parms.get("rtol", 1e-3), atol=solver_parms.get("atol", 1e-3),
                    max_step=solver_parms.get("max_step", np.inf), t_eval=tracker_parms["t_eval"],
                    events=True, event_capacity=64, device=device, **extra)
    if store_folder is not None:
        os.makedirs(store_folder, exist_ok=True)
        with hdf5lite.File(os.path.join(store_folder, "LMAHeureuxPorosityDiff_sweep.hdf5"), "w") as stored:
            stored.create_dataset("solutions", data=np.transpose(np.asarray(res.snapshots), (0, 2, 3, 1)))
            stored.create_dataset("times", data=res.t_eval)
            # next_eval: rows of `solutions` that hold data for a column (the rest is NaN: the column stopped early)
            for name in ("status", "nfev", "n_accepted", "n_rejected", "event_counts", "next_eval"):
                stored.create_dataset(name, data=np.asarray(getattr(res, name), dtype=np.int64))
            stored.create_dataset("t_reached", data=res.t)
            for k in ("sedimentationrate", "b", "DCO3", "Xstar", "Tstar"):
                stored.create_dataset("sweep_" + k, data=np.broadcast_to(np.asarray(pde_parms[k], float), res.t.shape))
            if extra:
                stored.create_dataset("sensitivities", data=np.transpose(np.asarray(res.sensitivities), (0, 1, 3, 4, 2)))
                stored.attrs.update({"sensitivity_directions": "\n".join(sensitivities.names)})
            stored.attrs.update({k: v for k, v in (solver_parms | tracker_parms).items() if k != "jac_sparsity"})
    return res


def Plot_results(last_field_sol, covered_time, depths, Xstar, store_folder):
    """Final depth profiles as a PDF (reference :185-205).  Plotting is cosmetic and needs
    matplotlib, which this image does not ship; without it the call is a no-op with a notice."""
    try:
        import matplotlib
        matplotlib.use("AGG")
        import matplotlib.pyplot as plt
    except ImportError:
        print("matplotlib is not installed: skipping Final_distributions.pdf")
        return
    fig, ax = plt.subplots()
    fig.suptitle(f"Distributions after {covered_time:.2e} years")
    x_cm = ScalarField.from_expression(depths, "x").data * Xstar
    for row, (marker, label) in enumerate((("v", "CA"), ("^", "CC"), (">", "cCa"), ("<", "cCO3"), ("o", "Phi"))):
        ax.plot(x_cm, last_field_sol[row], marker, ms=5, label=label)
    ax.set_xlabel("Depth (cm)")
    ax.set_ylabel("Compositions and concentrations (dimensionless)")
    ax.legend(loc="upper right")
    fig.savefig(store_folder + "Final_distributions.pdf", bbox_inches="tight")


if __name__ == "__main__":
    Plot_results(*integrate_equations(asdict(Solver()), asdict(Tracker()), asdict(Map_Scenario())))
