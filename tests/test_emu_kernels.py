"""Kernel control logic on the host: the batched Radau kernel (csrc/radau_batch.cu), the on-chip RK45 kernel
(csrc/rk45_persistent.cu) and the streaming RK45 path (csrc/rk45_streaming.cu) are compiled
for the host with g++ and run one thread block at a time by a small SIMT emulator (tests/emu/: one fiber per CUDA thread,
rendezvous at every barrier / warp collective / mbarrier wait; a missing barrier or a collective that not all named
lanes reach is reported instead of hanging).

This is test infrastructure, not a CPU path of the product: it checks indexing, halo exchange, barriers, slot service,
dense output and event location of a kernel BEFORE it is first launched on a GPU; arithmetic parity on the device stays
the job of the `-m gpu` tests.  Calibration: the default kernel under emulation reproduces SciPy RK45 exactly as it does
on the GPU (identical nfev, differences at the 1e-14 level)."""
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
np.seterr(all="ignore")


@pytest.fixture(scope="module")
def emu():
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    out = os.path.join(EMU, "_build")
    os.makedirs(out, exist_ok=True)
    srcs = [os.path.join(EMU, f) for f in ("emu_rk45.cc", "simt_emu.cc")]
    so = os.path.join(out, "libemu_rk45.so")
    done = subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-DMARLPDE_HOST_EMU", "-I", EMU, "-o", so] + srcs,
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    assert done.returncode == 0, done.stdout.decode()
    lib = C.CDLL(so)
    lib.emu_rk45.restype = C.c_int

    def run(variant, P, y, t_end, t_eval=(), events=False, first_step=1e-6, max_steps=0, state=None, capacity=16,
            quantum=None, flags=0):
        y = np.ascontiguousarray(y, dtype=np.float64).copy()
        P = np.ascontiguousarray(P)
        B, _, N = y.shape
        st = batch.make_state(B, 0.0, first_step) if state is None else state.copy()
        te = np.asarray(t_eval, dtype=np.float64)
        snap = np.full((B, max(1, te.size), 5, N), np.nan)
        ec = np.zeros((B, 7), np.int32)
        et = np.full((B, 7, capacity), np.nan)
        o = _cabi.RK45Options(t_bound=t_end, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=max_steps,
                              n_eval=te.size, event_capacity=capacity,
                              flags=flags | (_cabi.FLAG_EVENTS if events else 0) | (0 if quantum is None else _cabi.FLAG_QUEUE_LOCKS),
                              quantum=quantum or 0)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = lib.emu_rk45(variant, p(y), p(P), p(st), B, N, C.byref(o), p(te), p(snap), p(ec), p(et))
        assert rc == 0, f"emulated kernel {variant}: rc {rc} (deadlock or mismatched collective, see stderr)"
        return dict(y=y, state=st, snapshots=snap, event_counts=ec, event_times=et)
    return run


SCEN_A = {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}


def test_default_kernel_under_emulation_reproduces_scipy(emu):
    """Calibration of the emulator with the kernel that is validated on the GPU."""
    pde = oracle.default_scenario() | SCEN_A
    sol = oracle.integrate(pde, method="RK45", t_span=(0, 2e-4), t_eval=[2e-4], events=False, first_step=1e-6)
    for variant in (320,):
        res = emu(variant, mb.derive_column_params(pde), mb.initial_state(pde), 2e-4)
        assert res["state"]["status"][0] == 0 and res["state"]["nfev"][0] == sol.nfev, variant
        assert np.max(np.abs(res["y"][0] - sol.y.reshape(5, 200, -1)[:, :, -1])) <= 1e-12, variant


def test_quantum_major_work_items_are_bit_identical_to_whole_column_claims(emu, monkeypatch):
    """MARLPDE_FLAG_QUEUE_LOCKS: a column's step budget cut into quanta that are claimed quantum-major (the partly filled last
    round of a launch becomes 1 / n_quanta as long).  A quantum ends like a step budget and the next one resumes from the
    stored state, so the result must equal the whole-column claim bit for bit: 8 columns on 3 slots (every slot switches column
    at every quantum), 2 columns on 3 slots (a slot finds its column locked by another slot and retries), t_eval samples
    and events across quantum boundaries, a quantum that does not divide the budget, and the library's own choice."""
    pde = mb.sweep_lattice(oracle.default_scenario() | SCEN_A, 2, 2, 2)
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    te = [1e-4, 2.5e-4]
    whole = emu(320, P, y0, 1.0, t_eval=te, events=True, max_steps=100)
    for q in (7, 25, 100, 1000):
        part = emu(320, P, y0, 1.0, t_eval=te, events=True, max_steps=100, quantum=q)
        assert np.array_equal(part["y"], whole["y"]), q
        for k in ("t", "h_abs", "n_accepted", "n_rejected", "status", "next_eval"):
            assert np.array_equal(part["state"][k], whole["state"][k]), (q, k)
        # one extra K1 evaluation per resumed quantum, nothing else
        extra = part["state"]["nfev"] - whole["state"]["nfev"]
        assert np.all(extra == (100 + q - 1) // q - 1), (q, extra)
        assert np.array_equal(part["snapshots"], whole["snapshots"], equal_nan=True)
        assert np.array_equal(part["event_counts"], whole["event_counts"])
    two = emu(320, P[:2], y0[:2], 1.0, max_steps=60, quantum=9)
    ref = emu(320, P[:2], y0[:2], 1.0, max_steps=60)
    assert np.array_equal(two["y"], ref["y"]) and np.array_equal(two["state"]["t"], ref["state"]["t"])
    monkeypatch.setenv("EMU_SLOTS", "3")           # 8 columns on 3 slots: 2.67 rounds -> the library picks several quanta
    auto = emu(320, P, y0, 1.0, max_steps=640, quantum=0)
    ref = emu(320, P, y0, 1.0, max_steps=640)
    assert np.array_equal(auto["y"], ref["y"])
    assert np.all(auto["state"]["nfev"] > ref["state"]["nfev"])    # it did cut the budget
    assert np.array_equal(auto["state"]["n_accepted"], ref["state"]["n_accepted"])
    # no step budget (a sweep integrated to t_bound in one launch): 32 quanta, a column's last item runs without a limit
    whole = emu(320, P, y0, 2.5e-4, t_eval=te, events=True)
    for q in (2, 9):                      # 64 / 288 attempts in quanta: the rest of a column in its last item / all in quanta
        cut = emu(320, P, y0, 2.5e-4, t_eval=te, events=True, quantum=q)
        assert np.all(cut["state"]["status"] == 0) and np.all(cut["state"]["t"] == 2.5e-4), q
        assert np.array_equal(cut["y"], whole["y"]) and np.array_equal(cut["snapshots"], whole["snapshots"], equal_nan=True), q
        assert np.array_equal(cut["state"]["n_accepted"], whole["state"]["n_accepted"]), q
        assert np.array_equal(cut["event_counts"], whole["event_counts"]), q
        assert np.all(cut["state"]["nfev"][2:] > whole["state"]["nfev"][2:]), q       # the last 2 x 3 columns are cut ...
        assert np.array_equal(cut["state"]["nfev"][:2], whole["state"]["nfev"][:2]), q  # ... the first two claimed whole
    # the same split with a step budget (MARLPDE_FLAG_QUEUE_TAIL)
    ref = emu(320, P, y0, 1.0, max_steps=90)
    tail = emu(320, P, y0, 1.0, max_steps=90, quantum=8, flags=_cabi.FLAG_QUEUE_TAIL)
    assert np.array_equal(tail["y"], ref["y"]) and np.array_equal(tail["state"]["t"], ref["state"]["t"])
    assert np.array_equal(tail["state"]["nfev"][:2], ref["state"]["nfev"][:2]) and np.all(tail["state"]["nfev"][2:] > ref["state"]["nfev"][2:])


def test_event_bits_of_a_slot_that_idled_are_clean(emu):
    """Regression (found while the paired kernel shape was tried, r02z): a slot whose next work item belongs to a column
    locked by another slot idles for a few trips; if their number is odd, its first attempt on the new column used to find
    the PREVIOUS column's last predicate bits in the y_new buffer and reported spurious events.  Two columns on three
    slots in quanta of 7 attempts reproduce it (2 extra events before the fix); the start state makes four monitors fire
    within the first 60 attempts."""
    pde = mb.sweep_lattice(oracle.default_scenario() | SCEN_A, 1, 1, 2)
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    for f, frac, v in ((0, 0.25, -2e-5), (1, 0.30, -1e-5), (4, 0.75, 1.0 + 5e-6), (0, 0.60, -1.5e-5)):
        y0[:, f, int(frac * 200)] = v
    whole = emu(320, P, y0, 1.0, events=True, max_steps=60)
    assert whole["event_counts"].sum() >= 8
    for q in (7, 9):
        cut = emu(320, P, y0, 1.0, events=True, max_steps=60, quantum=q)
        assert np.array_equal(cut["event_counts"], whole["event_counts"]), q
        assert np.array_equal(cut["event_times"], whole["event_times"], equal_nan=True), q
        assert np.array_equal(cut["y"], whole["y"]), q


def test_time_varying_dPhi_instantiation_under_emulation(emu):
    """The kVarDPhi = true instantiation of the on-chip kernel (MARLPDE_FLAG_VAR_DPHI): a flagged column follows SciPy on
    the oracle's model variant (LHeureux_model.py:430), a plain column in the same launch is bit-identical to the default
    instantiation."""
    base = oracle.default_scenario() | SCEN_A
    var = base | {"time_varying_dPhi": True}
    P = np.concatenate([mb.derive_column_params(var), mb.derive_column_params(base)])
    Y = np.repeat(mb.initial_state(base), 2, 0)
    sol = oracle.integrate(var, method="RK45", t_span=(0, 2e-4), t_eval=[2e-4], events=False, first_step=1e-6)
    res = emu(320, P, Y, 2e-4, flags=_cabi.FLAG_VAR_DPHI)
    ref = emu(320, P[1:], Y[1:], 2e-4)
    assert res["state"]["nfev"][0] == sol.nfev and np.all(res["state"]["status"] == 0)
    assert np.max(np.abs(res["y"][0] - sol.y.reshape(5, 200, -1)[:, :, -1])) <= 1e-12
    assert np.array_equal(res["y"][1], ref["y"][0])
    assert np.max(np.abs(res["y"][0][4] - res["y"][1][4])) > 1e-8


# --------------------------------------------------------------------------------------- Radau kernel
@pytest.fixture(scope="module")
def emu_radau():
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    out = os.path.join(EMU, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemu_radau.so")
    srcs = [os.path.join(EMU, f) for f in ("emu_radau.cc", "simt_emu.cc")]
    subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-DMARLPDE_HOST_EMU", "-I", EMU, "-o", so] + srcs,
                   check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.emu_radau.restype = C.c_int
    lib.emu_radau_team.restype = C.c_int

    def run(P, y, t_end, t_eval=(), events=False, first_step=1e-6, team=False):
        y = np.ascontiguousarray(y, dtype=np.float64).copy()
        P = np.ascontiguousarray(P)
        B, _, N = y.shape
        st = batch.make_state(B, 0.0, first_step)
        te = np.asarray(t_eval, dtype=np.float64)
        snap = np.full((B, max(1, te.size), 5, N), np.nan)
        ec, et, stats = np.zeros((B, 7), np.int32), np.full((B, 7, 16), np.nan), np.zeros((B, 4), np.int64)
        o = _cabi.RK45Options(t_bound=t_end, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=0, n_eval=te.size,
                              event_capacity=16, flags=_cabi.FLAG_EVENTS if events else 0, quantum=0)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = (lib.emu_radau_team if team else lib.emu_radau)(p(y), p(P), p(st), B, N, C.byref(o), p(te), p(snap), p(stats), p(ec), p(et))
        assert rc == 0, f"emulated Radau kernel: rc {rc}"
        return dict(y=y, state=st, snapshots=snap, stats=stats, event_counts=ec, event_times=et)
    return run


def test_radau_kernel_under_emulation(emu_radau):
    """Scenario A to T* (the reference's regression case) and a lattice of five columns through the four warps of one CTA:
    the Radau kernel under emulation against SciPy Radau with the reference's sparsity."""
    pde = oracle.default_scenario() | SCEN_A
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    te = np.linspace(0, 1, 11)
    sol = oracle.integrate(pde, method="Radau", t_span=(0, 1), t_eval=te, events=False, first_step=1e-6,
                           jac_sparsity=oracle.jacobian_sparsity(200))
    want = np.moveaxis(sol.y.reshape(5, 200, -1), 2, 0)
    unit = 1e-3 + 1e-3 * np.abs(want)
    res = emu_radau(P, y0, 1.0, t_eval=te)
    assert res["state"]["status"][0] == 0 and 25 <= res["state"]["n_accepted"][0] <= 80
    assert np.max(np.abs(res["snapshots"][0] - want) / unit) <= 2.0      # two Radau codes at rtol = 1e-3
    lat = mb.sweep_lattice(oracle.default_scenario(), 1, 1, 5)
    Pl, yl = mb.derive_column_params(lat), mb.initial_state(lat)
    a = emu_radau(Pl, yl, 0.006, t_eval=[0.006], events=True, first_step=5e-7)
    assert np.all(a["state"]["status"] == 0)
    one = {k: (float(v[4]) if np.ndim(v) else v) for k, v in lat.items()}
    s4 = oracle.integrate(one, method="Radau", t_span=(0, 0.006), t_eval=[0.006], events=False, first_step=5e-7,
                          jac_sparsity=oracle.jacobian_sparsity(200)).y.reshape(5, 200)
    assert np.max(np.abs(a["y"][4] - s4) / (1e-3 + 1e-3 * np.abs(s4))) <= 1.0


def test_radau_team_kernel_under_emulation(emu_radau):
    """The TEAM shape of the Radau kernel (two warps per column, a CTA each: split RHS / element-wise passes / Jacobian,
    the two factorisation chains on one warp each, team-wide reductions, block barriers) against the one-warp shape: the
    emulator reports a barrier that not every thread reaches or a deadlock; the two shapes must take the same steps, LU
    and Newton counts and events, with states equal up to the order of the norm reductions."""
    pde = oracle.default_scenario() | SCEN_A
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    te = np.linspace(0, 1, 6)
    a, b = emu_radau(P, y0, 1.0, t_eval=te), emu_radau(P, y0, 1.0, t_eval=te, team=True)
    assert np.array_equal(a["state"], b["state"]) or (a["state"]["n_accepted"] == b["state"]["n_accepted"]).all()
    assert np.array_equal(a["stats"], b["stats"])
    assert np.max(np.abs(a["snapshots"] - b["snapshots"])) <= 1e-10
    lat = mb.sweep_lattice(oracle.default_scenario(), 1, 1, 3)          # three columns through the team's queue, events on
    Pl, yl = mb.derive_column_params(lat), mb.initial_state(lat)
    a = emu_radau(Pl, yl, 0.03, t_eval=[0.03], events=True, first_step=5e-7)
    b = emu_radau(Pl, yl, 0.03, t_eval=[0.03], events=True, first_step=5e-7, team=True)
    assert np.array_equal(a["stats"], b["stats"]) and np.array_equal(a["event_counts"], b["event_counts"])
    assert a["event_counts"].sum() >= 5
    assert np.max(np.abs(a["y"] - b["y"])) <= 1e-9
    assert np.nanmax(np.abs(a["event_times"] - b["event_times"])) <= 1e-10


# ----------------------------------------------------------------------------------------- BDF kernel
def exact_sparsity(N):
    """The block-tridiagonal structure (cell-major 5x5 blocks) as a field-major sparsity pattern for SciPy."""
    import scipy.sparse as sp
    cells = np.arange(5 * N) % N
    return sp.csr_matrix((np.abs(cells[:, None] - cells[None, :]) <= 1).astype(float))


@pytest.fixture(scope="module")
def emu_bdf():
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    out = os.path.join(EMU, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemu_bdf.so")
    srcs = [os.path.join(EMU, f) for f in ("emu_bdf.cc", "simt_emu.cc")]
    subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-DMARLPDE_HOST_EMU", "-I", EMU, "-o", so] + srcs,
                   check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.emu_bdf.restype = C.c_int

    def run(P, y, t_end, t_eval=(), events=False, first_step=1e-6, tol=1e-3, jac="analytic"):
        y = np.ascontiguousarray(y, dtype=np.float64).copy()
        P = np.ascontiguousarray(P)
        B, _, N = y.shape
        st = batch.make_state(B, 0.0, first_step)
        te = np.asarray(t_eval, dtype=np.float64)
        snap = np.full((B, max(1, te.size), 5, N), np.nan)
        ec, et, stats = np.zeros((B, 7), np.int32), np.full((B, 7, 16), np.nan), np.zeros((B, 4), np.int64)
        o = _cabi.RK45Options(t_bound=t_end, rtol=tol, atol=tol, max_step=float("inf"), max_steps=0, n_eval=te.size,
                              event_capacity=16, flags=(_cabi.FLAG_EVENTS if events else 0) |
                              (_cabi.FLAG_JAC_FD if jac == "fd" else 0), quantum=0)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = lib.emu_bdf(p(y), p(P), p(st), B, N, C.byref(o), p(te), p(snap), p(stats), p(ec), p(et))
        assert rc == 0, f"emulated BDF kernel: rc {rc}"
        return dict(y=y, state=st, snapshots=snap, stats=stats, event_counts=ec, event_times=et)
    return run


def test_bdf_kernel_under_emulation_is_scipy_bdf_step_for_step(emu_bdf):
    """The BDF kernel (csrc/bdf_batch.cu) restates scipy/integrate/_ivp/bdf.py; handed the SAME Jacobian structure (the
    block-tridiagonal pattern instead of the reference's 27 diagonals, which drop d(CA,CC)/dPhi) SciPy's BDF takes the same
    steps: identical Jacobian and LU counts, one Newton iteration per SciPy RHS call, states equal to a small fraction of
    the tolerance — at rtol = 1e-3 and 1e-6, scenario A to T* (the reference's regression case) with dense output."""
    pde = oracle.default_scenario() | SCEN_A
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    for tol, te, gate, jac in ((1e-3, np.linspace(0, 1, 6), 1e-3, "fd"), (1e-3, np.linspace(0, 1, 6), 1e-3, "analytic"),
                               (1e-6, np.array([0.0, 0.1]), 1e-2, "fd")):
        sol = oracle.integrate(pde, method="BDF", t_span=(0, te[-1]), t_eval=te, events=False, first_step=1e-6, rtol=tol,
                               atol=tol, jac_sparsity=exact_sparsity(200))
        res = emu_bdf(P, y0, te[-1], t_eval=te, tol=tol, jac=jac)
        assert res["state"]["status"][0] == 0
        assert res["stats"][0, 0] == sol.njev and res["stats"][0, 1] == sol.nlu
        assert res["stats"][0, 2] == sol.nfev - 1                      # bdf.py: one fun call per Newton iteration + f(t0, y0)
        assert res["state"]["nfev"][0] == sol.nfev + (6 * sol.njev if jac == "fd" else 0)   # + f0 and 5 colours per Jacobian
        want = np.moveaxis(sol.y.reshape(5, 200, -1), 2, 0)
        assert np.max(np.abs(res["snapshots"][0] - want) / (tol + tol * np.abs(want))) <= gate


def test_bdf_kernel_events_and_lattice_under_emulation(emu_bdf):
    """Event monitors on the BDF dense output (default scenario: the porosity crosses 1 near t = 0.026, then max W changes
    sign) against SciPy BDF's events; five lattice columns through the four warps of one CTA."""
    pde = oracle.default_scenario()
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    sol = oracle.integrate(pde, method="BDF", t_span=(0, 0.0275), t_eval=[0.0275], events=True, first_step=5e-7,
                           jac_sparsity=exact_sparsity(200))
    res = emu_bdf(P, y0, 0.0275, t_eval=[0.0275], events=True, first_step=5e-7)
    assert [len(e) for e in sol.t_events] == list(res["event_counts"][0])
    for k in (4, 6):
        assert len(sol.t_events[k]) >= 1
        assert np.max(np.abs(res["event_times"][0, k, :len(sol.t_events[k])] - sol.t_events[k])) <= 1e-6
    lat = mb.sweep_lattice(oracle.default_scenario(), 1, 1, 5)
    Pl, yl = mb.derive_column_params(lat), mb.initial_state(lat)
    a = emu_bdf(Pl, yl, 0.006, t_eval=[0.006], first_step=5e-7)
    assert np.all(a["state"]["status"] == 0)
    one = {k: (float(v[4]) if np.ndim(v) else v) for k, v in lat.items()}
    s4 = oracle.integrate(one, method="BDF", t_span=(0, 0.006), t_eval=[0.006], events=False, first_step=5e-7,
                          jac_sparsity=exact_sparsity(200))
    assert a["stats"][4, 1] == s4.nlu
    assert np.max(np.abs(a["y"][4] - s4.y.reshape(5, 200)) / (1e-3 + 1e-3 * np.abs(s4.y.reshape(5, 200)))) <= 0.01


# ------------------------------------------------------------------- streaming path (large depth grids)
@pytest.fixture(scope="module")
def emu_stream():
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    out = os.path.join(EMU, "_build")
    os.makedirs(out, exist_ok=True)
    srcs = [os.path.join(EMU, f) for f in ("emu_stream.cc", "simt_emu.cc")]
    so = os.path.join(out, "libemu_stream.so")
    subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-DMARLPDE_HOST_EMU", "-I", EMU, "-o", so] + srcs,
                   check=True, capture_output=True)
    lib = C.CDLL(so)
    lib.emu_rk45_stream.restype = C.c_int

    def run(P, y, t_end, t_eval, first_step, attempts, state=None, events=False, counts=None, times=None, flags=0,
            tile=None):
        # the launcher reads the window size switch per call
        if tile:
            os.environ["MARLPDE_RK45_TILE"] = tile
        else:
            os.environ.pop("MARLPDE_RK45_TILE", None)
        y = np.ascontiguousarray(y, dtype=np.float64).copy()
        P = np.ascontiguousarray(P)
        B, _, N = y.shape
        st = batch.make_state(B, 0.0, first_step) if state is None else state.copy()
        te = np.asarray(t_eval, dtype=np.float64)
        snap = np.full((B, max(1, te.size), 5, N), np.nan)
        ec = np.zeros((B, 7), np.int32) if counts is None else counts.copy()
        et = np.full((B, 7, 16), np.nan) if times is None else times.copy()
        o = _cabi.RK45Options(t_bound=t_end, rtol=1e-3, atol=1e-3, max_step=float("inf"), max_steps=attempts,
                              n_eval=te.size, event_capacity=16, flags=flags | (_cabi.FLAG_EVENTS if events else 0), quantum=0)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = lib.emu_rk45_stream(p(y), p(P), p(st), B, N, C.byref(o), p(te), p(snap), C.c_longlong(attempts), p(ec), p(et))
        assert rc == 0, f"emulated streaming launcher: rc {rc}"
        return dict(y=y, state=st, snapshots=snap, event_counts=ec, event_times=et)
    return run


@pytest.mark.parametrize("n_cells,ncol", [(16, 2), (641, 2), (1257, 1)])
def test_streaming_launcher_under_emulation_reproduces_scipy(emu_stream, n_cells, ncol):
    """csrc/rk45_streaming.cu with its own launcher (init / K1 / tile_attempt / prepare / copyback / finish), every launch
    run block by block: ragged last windows, batches of 16 attempts resumed from the column state as the host driver
    does (csrc/cabi.cu rk45_integrate_streaming) — the GPU test test_streaming_path_matches_scipy at a shorter t_end."""
    pde = oracle.default_scenario() | SCEN_A | {"N": n_cells}
    scale = min(1.0, (200 / n_cells) ** 2)
    t_end, fs = 60 * 2.6e-6 * scale, 1e-6 * scale
    te = [0.0, 0.4 * t_end, t_end]
    P, y0 = np.repeat(mb.derive_column_params(pde), ncol), np.repeat(mb.initial_state(pde), ncol, 0)
    sol = oracle.integrate(pde, method="RK45", t_span=(0, t_end), t_eval=te, events=False, first_step=fs)
    want = sol.y.reshape(5, n_cells, -1)
    r = emu_stream(P, y0, t_end, te, fs, 16)
    while np.any((r["state"]["status"] == 1) | (r["state"]["status"] == 2)):
        nxt = emu_stream(P, r["y"], t_end, te, fs, 16, state=r["state"])
        keep = np.isnan(nxt["snapshots"])
        nxt["snapshots"][keep] = r["snapshots"][keep]
        r = nxt
    assert np.all(r["state"]["status"] == 0) and np.all(r["state"]["t"] == t_end) and np.all(r["state"]["next_eval"] == 3)
    assert np.all(r["state"]["nfev"] == sol.nfev), (r["state"]["nfev"], sol.nfev)
    assert np.max(np.abs(r["y"][0] - want[:, :, -1])) <= 1e-12
    assert np.max(np.abs(r["snapshots"][0] - np.moveaxis(want, 2, 0))) <= 1e-12
    assert np.array_equal(r["y"][0], r["y"][-1])


@pytest.mark.parametrize("n_cells", [16, 628, 1256, 1884, 1300])
def test_tile_kernel_window_sizes_agree(emu_stream, n_cells):
    """The tile kernel's two window sizes, each selected explicitly: 640-cell windows (320 threads, 628 owned cells) and
    256-cell windows (128 threads, 244 owned cells).  Window clipping at both column ends, a column that ends exactly on
    a window boundary, one-window columns and a sampled step.  The error norm adds one partial sum per window in window
    order, so the step sizes of the two window sizes may differ in their last bits: same decisions, states equal to
    round-off.  The launcher picks the small windows for every size here (one column on 148 SMs): bit for bit."""
    pde = oracle.default_scenario() | SCEN_A | {"N": n_cells}
    scale = min(1.0, (200 / n_cells) ** 2)
    fs = 1e-6 * scale
    te = [0.0, 4 * fs, 1.0]
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    y0 = y0 * (1 + 0.01 * np.sin(np.arange(n_cells) * 0.37))          # a profile, so that misplaced rows would show
    large = emu_stream(P, y0, 1.0, te, fs, 12, tile="large")
    small = emu_stream(P, y0, 1.0, te, fs, 12, tile="small")
    auto = emu_stream(P, y0, 1.0, te, fs, 12)
    assert large["state"]["n_accepted"][0] >= 8 and large["state"]["next_eval"][0] == 2
    for k in ("n_accepted", "n_rejected", "nfev", "status", "next_eval"):
        assert np.array_equal(large["state"][k], small["state"][k]), k
    assert abs(large["state"]["t"][0] - small["state"]["t"][0]) <= 1e-12 * large["state"]["t"][0]
    assert np.max(np.abs(large["y"] - small["y"])) <= 1e-12
    assert np.max(np.abs(large["snapshots"][:, :2] - small["snapshots"][:, :2])) <= 1e-12
    assert np.array_equal(auto["state"], small["state"]) and np.array_equal(auto["y"], small["y"])
    assert np.array_equal(auto["snapshots"][:, :2], small["snapshots"][:, :2])


@pytest.mark.parametrize("n_cells", [16, 1300])
def test_streaming_events_replay_and_locate_under_emulation(emu_stream, n_cells):
    """Event monitors on the streaming path: per-window predicate bits, detection in the prepare kernel, replay of the
    step with K3..K6 stored, Brent location by the column's first CTA.  Counts and root times equal SciPy's; a run cut
    into batches of 16 attempts (a batch may end between detection and location; 5 for the 16-cell grid) finds every event exactly once; the
    trajectory does not depend on monitoring."""
    pde = oracle.default_scenario() | SCEN_A | {"N": n_cells}
    scale = min(1.0, (200 / n_cells) ** 2)
    t_end, fs = 90 * 2.6e-6 * scale, 1e-6 * scale
    y0 = mb.initial_state(pde)
    pick = lambda frac: min(n_cells - 1, int(frac * n_cells))
    y0[0, 0, pick(0.25)] = -2e-5 * scale
    y0[0, 1, pick(0.30)] = -1e-5 * scale
    y0[0, 4, pick(0.75)] = 1.0 + 5e-6 * scale
    sol = oracle.integrate(pde, method="RK45", t_span=(0, t_end), t_eval=[0, t_end], events=True, y0=y0[0], first_step=fs)
    want = [len(e) for e in sol.t_events]
    assert sum(want) >= 3, want
    P = mb.derive_column_params(pde)
    plain = emu_stream(P, y0, t_end, [t_end], fs, 200)
    assert plain["state"]["status"][0] == 0
    per_call = 5 if n_cells < 100 else 16
    r = emu_stream(P, y0, t_end, [t_end], fs, per_call, events=True)
    times = [list(r["event_times"][0, k, :r["event_counts"][0, k]]) for k in range(7)]
    hops = 1
    while r["state"]["status"][0] in (1, 2):
        r = emu_stream(P, r["y"], t_end, [t_end], fs, per_call, state=r["state"], events=True)
        for k in range(7):
            times[k] += list(r["event_times"][0, k, :r["event_counts"][0, k]])
        hops += 1
    assert hops >= 3 and r["state"]["status"][0] == 0
    assert [len(t) for t in times] == want
    for k in range(7):
        assert np.allclose(np.sort(times[k]), sol.t_events[k], rtol=0, atol=1e-12)
    assert np.array_equal(r["y"], plain["y"]) and r["state"]["nfev"][0] == plain["state"]["nfev"][0] == sol.nfev
