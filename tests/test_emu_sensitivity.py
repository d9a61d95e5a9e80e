"""Forward sensitivities of the BDF kernel (csrc/bdf_batch.cu, bdf_kernel<., ., true>) under the SIMT emulator
(tests/emu/emu_bdf_sens.cc): the state's path is bit-identical to the kernel without sensitivities (tests/emu/emu_bdf.cc),
and s = dy/d eps agrees with central differences of the emulated integration itself.

Test infrastructure, not a CPU path of the product: the emulator runs the kernel source compiled for the host."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import lheureux_oracle as oracle
import marlpde_b200 as mb
from marlpde_b200 import _cabi, batch
from conftest import ROOT

EMU = os.path.join(ROOT, "tests", "emu")
SCEN_A = {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
np.seterr(all="ignore")


def _build(name):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    out = os.path.join(EMU, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, f"lib{name}.so")
    srcs = [os.path.join(EMU, f) for f in (f"{name}.cc", "simt_emu.cc")]
    subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-DMARLPDE_HOST_EMU", "-I", EMU, "-o", so] + srcs,
                   check=True, capture_output=True)
    lib = C.CDLL(so)
    getattr(lib, name).restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def emu():
    """run(P, y, t_end, ..., sens=None): the emulated BDF kernel; with sens = (directions, w) the sensitivity build."""
    plain, withs = _build("emu_bdf"), _build("emu_bdf_sens")

    def run(P, y, t_end, t_eval=(), events=False, first_step=1e-6, tol=1e-3, max_steps=0, state=None, sens=None,
            sens_y=None, jac="analytic"):
        y = np.ascontiguousarray(y, dtype=np.float64).copy()
        P = np.ascontiguousarray(P)
        B, _, N = y.shape
        st = batch.make_state(B, 0.0, first_step) if state is None else np.array(state, copy=True)
        te = np.asarray(t_eval, dtype=np.float64)
        snap = np.full((B, max(1, te.size), 5, N), np.nan)
        ec, et, stats = np.zeros((B, 7), np.int32), np.full((B, 7, 16), np.nan), np.zeros((B, 4), np.int64)
        o = _cabi.RK45Options(t_bound=t_end, rtol=tol, atol=tol, max_step=float("inf"), max_steps=max_steps,
                              n_eval=te.size, event_capacity=16, flags=(_cabi.FLAG_EVENTS if events else 0) |
                              (_cabi.FLAG_JAC_FD if jac == "fd" else 0), quantum=0)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        out = dict(y=y, state=st, snapshots=snap, stats=stats, event_counts=ec, event_times=et)
        if sens is None:
            rc = plain.emu_bdf(p(y), p(P), p(st), B, N, C.byref(o), p(te), p(snap), p(stats), p(ec), p(et))
        else:
            nd = sens.n_dirs
            s = np.ascontiguousarray(sens.w if sens_y is None else sens_y, dtype=np.float64).copy()
            ssnap = np.full((B, nd, max(1, te.size), 5, N), np.nan)
            sstats = np.zeros((B, 3), np.int64)
            atol_s = sens.atol(tol)
            rc = withs.emu_bdf_sens(p(y), p(P), p(st), B, N, C.byref(o), p(te), p(snap), p(stats), p(ec), p(et), nd,
                                    p(sens.params_pm), p(sens.inv2sigma), p(atol_s), p(s), p(ssnap), p(sstats))
            out.update(sens_y=s, sens_snap=ssnap, sens_stats=sstats)
        assert rc == 0, f"emulated BDF kernel: rc {rc}"
        return out
    return run


def _same_state_path(a, b):
    for k in ("y", "snapshots", "stats", "event_counts"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert a["state"].tobytes() == b["state"].tobytes()
    assert np.array_equal(a["event_times"], b["event_times"], equal_nan=True)


def test_state_path_is_bit_identical_with_sensitivities(emu):
    """The central invariant: with P = 2 directions the state's y, column state, counters, snapshots, event counts and
    event times are bit-identical to the kernel without sensitivities — scenario A on 33 cells to t = 0.0275 with
    events, and the lattice columns of the BDF emulator test."""
    pde = oracle.default_scenario() | SCEN_A | {"N": 33}
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    sd = mb.sensitivity_directions(pde, ["k2", "PhiIni"])
    te = [0.0, 0.01, 0.0275]
    a = emu(P, y0, 0.0275, t_eval=te, events=True, first_step=5e-7)
    b = emu(P, y0, 0.0275, t_eval=te, events=True, first_step=5e-7, sens=sd)
    _same_state_path(a, b)
    assert a["state"]["status"][0] == 0 and np.all(np.isfinite(b["sens_y"]))
    lat = mb.sweep_lattice(oracle.default_scenario(), 1, 1, 5)
    Pl, yl = mb.derive_column_params(lat), mb.initial_state(lat)
    sl = mb.sensitivity_directions(lat, ["DCO3", "b"])
    a = emu(Pl, yl, 0.006, t_eval=[0.006], first_step=5e-7)
    b = emu(Pl, yl, 0.006, t_eval=[0.006], first_step=5e-7, sens=sl)
    _same_state_path(a, b)
    assert np.all(b["sens_stats"][:, 0] > 0)


def _S_direction(pde):
    S, D0Ca = pde["sedimentationrate"], pde["D0Ca"]
    return {"sedimentationrate": 1.0, "Xstar": -D0Ca / S ** 2, "Tstar": -2.0 * D0Ca / S ** 3}


DIRS = ["k2", "b", "DCO3", "PhiIni"]


def _fd_of_integration(emu, pde, direction, rel, t_end, tol, first_step):
    """Central difference of the emulated (state-only) integration along `direction` with step rel * pbar."""
    name, coef = (direction, {direction: 1.0}) if isinstance(direction, str) else ("S", direction)
    pbar = min(abs(pde[k]) / abs(c) for k, c in coef.items() if pde[k] != 0 and c != 0)
    h = rel * pbar
    ys = []
    for sgn in (1.0, -1.0):
        q = dict(pde)
        for k, c in coef.items():
            q[k] = pde[k] + sgn * h * c
        ys.append(emu(mb.derive_column_params(q), mb.initial_state(q), t_end, tol=tol, first_step=first_step)["y"][0])
    return (ys[0] - ys[1]) / (2 * h)


T_TIGHT = 0.004


@pytest.fixture(scope="module")
def tight(emu):
    """Scenario A on 33 cells to t = 0.004 at rtol = atol = 1e-9: sensitivities along k2, b, DCO3, PhiIni and the
    consistent S direction, and the same at the reference tolerance 1e-3."""
    pde = oracle.default_scenario() | SCEN_A | {"N": 33}
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    sd = mb.sensitivity_directions(pde, DIRS + [_S_direction(pde)])
    res = {tol: emu(P, y0, T_TIGHT, t_eval=[0.0, T_TIGHT], tol=tol, first_step=1e-7, sens=sd) for tol in (1e-9, 1e-3)}
    return pde, sd, res


def test_sensitivities_match_central_differences_of_the_integration(emu, tight):
    """At rtol = atol = 1e-9 s(T) along k2, b, DCO3, PhiIni and the consistent S direction matches the central difference
    of the emulated integration itself (step 1e-3 pbar: truncation ~1e-6, step-control noise ~tol / 1e-3) to 1e-4 of
    max |s|."""
    pde, sd, res = tight
    r = res[1e-9]
    assert r["state"]["status"][0] == 0
    for k, d in enumerate(DIRS + [_S_direction(pde)]):
        fd = _fd_of_integration(emu, pde, d, 1e-3, T_TIGHT, 1e-9, 1e-7)
        s = r["sens_y"][0, k]
        err = np.max(np.abs(s - fd)) / np.max(np.abs(s))
        assert err <= 1e-4, (sd.names[k], err)


def test_sensitivities_at_the_reference_tolerance(tight):
    """At rtol = atol = 1e-3 (the reference's tolerances) s(T) agrees with the tight-tolerance s to 3 tolerance units
    (atol_s + rtol |s|, atol_s = atol / pbar).  Measured: 0.02-1.5 units over the five directions, while the state itself
    deviates 0.7 units.  The cause is that s is integrated on the state's step sequence WITHOUT error control (errconS =
    false): its local truncation error is not bounded by the step-size controller, only inherited through the state's
    step sizes, so it is of the order of the state's own global error, somewhat larger for the directions whose forcing
    is largest where the state changes fastest (PhiIni, S).  The gate is twice the measured maximum."""
    pde, sd, res = tight
    a, b = res[1e-9], res[1e-3]
    at = sd.atol(1e-3)
    for k in range(sd.n_dirs):
        s9, s3 = a["sens_y"][0, k], b["sens_y"][0, k]
        dev = np.max(np.abs(s3 - s9) / (at[0, k] + 1e-3 * np.abs(s9)))
        assert dev <= 3.0, (sd.names[k], dev)
    assert b["sens_stats"][0, 2] == 0


def test_t_eval_sample_at_t0_is_w(tight):
    """The t_eval sample at the start time is w = dy0 / d eps itself, bit for bit."""
    pde, sd, res = tight
    for r in res.values():
        assert r["state"]["next_eval"][0] == 2
        assert np.array_equal(r["sens_snap"][0, :, 0], sd.w[0])


def test_budget_cut_and_resumed_run_keeps_the_state_path(emu):
    """A run cut by max_steps and resumed with sens_y has the same state as the same cut-and-resumed run without
    sensitivities (both restart at order 1), and its s ends close to an uncut run's."""
    pde = oracle.default_scenario() | SCEN_A | {"N": 33}
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    sd = mb.sensitivity_directions(pde, ["k2", "DCO3"])
    kw = dict(t_eval=[0.002, 0.005], first_step=1e-7)
    a1 = emu(P, y0, 0.005, max_steps=15, **kw)
    b1 = emu(P, y0, 0.005, max_steps=15, sens=sd, **kw)
    _same_state_path(a1, b1)
    assert a1["state"]["status"][0] == _cabi.STATUS_STEP_BUDGET
    a2 = emu(P, a1["y"], 0.005, state=a1["state"], **kw)
    b2 = emu(P, b1["y"], 0.005, state=b1["state"], sens=sd, sens_y=b1["sens_y"], **kw)
    for k in ("y", "stats", "event_counts"):
        assert np.array_equal(a2[k], b2[k], equal_nan=True), k
    assert a2["state"].tobytes() == b2["state"].tobytes() and a2["state"]["status"][0] == 0
    whole = emu(P, y0, 0.005, sens=sd, **kw)
    at = sd.atol(1e-3)
    for k in range(sd.n_dirs):
        dev = np.max(np.abs(b2["sens_y"][0, k] - whole["sens_y"][0, k]) / (at[0, k] + 1e-3 * np.abs(whole["sens_y"][0, k])))
        assert dev <= 3.0, (sd.names[k], dev)
