"""Host logic: per-column constants, sweep lattice, HDF5 writer/reader, C-ABI surface (no compute)."""
import ctypes
import os
import re

import numpy as np
import pytest

import lheureux_oracle as oracle
import marlpde_b200 as mb
from marlpde_b200 import _cabi, hdf5lite
from conftest import ROOT

np.seterr(all="ignore")


def test_column_params_equal_oracle_and_reference(rhs_golden):
    g, meta = rhs_golden
    for name, pde in meta.items():
        P = mb.derive_column_params(pde)
        assert P.shape == (1,)
        po = oracle.kernel_params(pde)
        for k in ("presum", "rhorat", "Da", "lambda_", "dCa", "dCO3", "delta", "KRat", "nu1", "nu2", "m1", "m2",
                  "n1", "n2", "dPhi_fixed", "dx", "delta_x", "Peclet_min", "Peclet_max"):
            assert P[k][0] == po[oracle.P_IDX[k]], (name, k)
        assert P["inv_dx2"][0] == po[oracle.P_IDX["dx_m2"]]
        assert (P["mask_lo"][0], P["mask_hi"][0]) == (po[oracle.P_IDX["mask_lo"]], po[oracle.P_IDX["mask_hi"]])
        assert np.array_equal(P["bc_top"][0], po[:5])
        assert bool(P["FV_switch"][0]) == bool(pde["FV_switch"])
        ref = g[f"{name}/derived"]        # the reference's own __init__ values
        assert np.array_equal([P[k][0] for k in ("presum", "rhorat", "Da", "lambda_", "dCa", "dCO3", "delta",
                                                 "KRat", "nu1", "nu2", "dPhi_fixed", "delta_x")], ref[:12])


def test_sweep_lattice_is_vectorised_map_scenario():
    base = oracle.default_scenario()
    pde = mb.sweep_lattice(base, 4, 3, 2)
    P = mb.derive_column_params(pde)
    y0 = mb.initial_state(pde)
    assert P.shape == (24,) and y0.shape == (24, 5, 200)
    # column c = (i*3 + j)*2 + k ; spot-check one column against the scalar derivation
    i, j, k = 2, 1, 1
    c = (i * 3 + j) * 2 + k
    raw = {kk: base[kk] for kk in base}
    raw.update(sedimentationrate=0.09 + 0.02 * i / 3, b=(4 + 2 * j / 2) / 1e4, DCO3=245 + 55 * k / 1)
    raw["Xstar"] = raw["D0Ca"] / raw["sedimentationrate"]
    raw["Tstar"] = raw["Xstar"] / raw["sedimentationrate"]
    one = mb.derive_column_params(raw)
    for name in P.dtype.names:
        assert np.array_equal(P[name][c], one[name][0]), name
    assert np.all(P["mask_hi"] > P["mask_lo"])


def test_params_validation():
    pde = oracle.default_scenario()
    bad = dict(pde)
    del bad["KC"]
    with pytest.raises(KeyError):
        mb.derive_column_params(bad)
    with pytest.raises(ValueError):
        mb.derive_column_params(pde | {"m1": 0.0})


def test_hdf5_roundtrip_layout_of_the_reference_driver(tmp_path):
    """Same dataset names/shapes/attrs as Evolve_scenario.py:170-178."""
    p = tmp_path / "LMAHeureuxPorosityDiff.hdf5"
    sol = np.arange(5 * 7 * 3, dtype=float).reshape(5, 7, 3)
    attrs = {"method": "RK45", "rtol": 1e-3, "N": 200, "dense_output": False, "t_span": (0, 1),
             "t_eval": np.linspace(0, 1, 3), "cCa0": np.float64(0.499), "first_step": 1e-6}
    with hdf5lite.File(p, "w") as f:
        f.create_dataset("solutions", data=sol)
        f.create_dataset("times", data=np.linspace(0, 1, 3))
        for k in range(7):
            f.create_dataset(f"event_{k}", data=np.array([]) if k != 6 else np.array([0.25, 0.5]))
        f.attrs.update(attrs)
    raw = p.read_bytes()
    assert raw[:8] == b"\x89HDF\r\n\x1a\n" and raw[8] == 0            # superblock v0
    assert int.from_bytes(raw[40:48], "little") == len(raw)            # end-of-file address
    with hdf5lite.File(p, "r") as f:
        assert sorted(f.keys()) == sorted(["solutions", "times"] + [f"event_{k}" for k in range(7)])
        assert np.array_equal(f["solutions"][:, :, -1], sol[:, :, -1])
        assert f.get("solutions").shape == (5, 7, 3)
        assert f["event_0"].shape == (0,) and np.array_equal(f["event_6"][:], [0.25, 0.5])
        assert f.attrs["method"] == "RK45" and f.attrs["N"] == 200 and f.attrs["dense_output"] == False  # noqa: E712
        assert np.array_equal(f.attrs["t_span"], [0, 1]) and f.attrs["first_step"] == 1e-6
        assert f.get("nope") is None
        with pytest.raises(OSError):
            f.attrs.update({"x": 1})


def test_cabi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "marlpde_b200.h")).read()
    declared = set(re.findall(r"^(?:int|size_t|const char\*)\s+(marlpde_[a-z0-9_]+)\s*\(", header, flags=re.M))
    assert declared == set(_cabi.SYMBOLS), declared ^ set(_cabi.SYMBOLS)
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    L = _cabi.lib()
    assert L.marlpde_abi_version() == 2
    assert L.marlpde_struct_size(0) == _cabi.PARAMS_DTYPE.itemsize == 232
    assert L.marlpde_struct_size(2) == _cabi.STATE_DTYPE.itemsize == 48
    assert L.marlpde_struct_size(9) == -1
    assert L.marlpde_rk45_max_cells() == 640
    assert L.marlpde_rk45_columns_per_cta(200) == 3
    assert L.marlpde_rk45_columns_per_cta(640) == 1 and L.marlpde_rk45_columns_per_cta(639) == 1
    assert L.marlpde_rk45_columns_per_cta(641) == 0 and L.marlpde_rk45_columns_per_cta(16) == 0


_NO_DEVICE_CHECK = """
import pytest
import lheureux_oracle as oracle
import marlpde_b200 as mb
from marlpde_b200 import _cabi
assert _cabi.lib().marlpde_device_count() == 0
pde = oracle.default_scenario()
with pytest.raises(_cabi.MarlpdeError, match="no CUDA device"):
    mb.rhs_batch(mb.initial_state(pde), mb.derive_column_params(pde))
with pytest.raises(_cabi.MarlpdeError, match="no CUDA device"):
    mb.integrate_rk45_batch(mb.initial_state(pde), mb.derive_column_params(pde), t_span=(0, 1e-4))
"""


def test_no_device_fails_loudly():
    """The product has no CPU fallback: on a box without a GPU compute calls must raise.  Runs in a child process
    with every device hidden (CUDA_VISIBLE_DEVICES=""), so it checks the same on a machine that has one."""
    import subprocess
    import sys
    path = [os.path.join(ROOT, "integrating-diagenetic-equations-using-python_b200"), os.path.join(ROOT, "oracle"),
            os.environ.get("PYTHONPATH", "")]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=os.pathsep.join(p for p in path if p))
    done = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECK], env=env, capture_output=True, text=True, timeout=300)
    assert done.returncode == 0, done.stderr[-2000:]


def test_argument_validation_before_any_device_work():
    pde = oracle.default_scenario()
    P, y0 = mb.derive_column_params(pde), mb.initial_state(pde)
    with pytest.raises(ValueError, match="first_step"):
        mb.integrate_rk45_batch(y0, P, first_step=0.0)
    with pytest.raises(ValueError, match="exceeds bounds"):
        mb.integrate_rk45_batch(y0, P, first_step=2.0)
    with pytest.raises(ValueError, match="not within"):
        mb.integrate_rk45_batch(y0, P, t_eval=[0.0, 2.0])
    with pytest.raises(ValueError, match="sorted"):
        mb.integrate_rk45_batch(y0, P, t_eval=[0.5, 0.25])
    with pytest.raises(ValueError):
        mb.rhs_batch(y0[:, :4], P)
    opts = _cabi.RK45Options(t_bound=1.0, rtol=1e-3, atol=1e-3, max_step=float("inf"))
    # the on-chip kernel's device entry point refuses grids that do not fit shared memory ...
    rc = _cabi.lib().marlpde_rk45_integrate_dev(None, None, None, 1, 1000, ctypes.byref(opts), None, None, None, None,
                                                None, None)
    assert rc == -4 and b"n_cells" in _cabi.lib().marlpde_last_error()
    # ... the host entry point routes them to the streaming path, which validates its own arguments
    rc = _cabi.lib().marlpde_rk45_integrate(None, None, None, 1, 1000, ctypes.byref(opts), None, None, None, None, 0)
    assert rc == -1 and b"NULL" in _cabi.lib().marlpde_last_error()
    # events are monitored on the streaming path too; the entry point without event outputs says which one to call
    opts.flags = _cabi.FLAG_EVENTS
    opts.max_steps = 8
    rc = _cabi.lib().marlpde_rk45_stream_integrate_dev(None, None, None, 1, 1000, ctypes.byref(opts), None, None, None, 0, None)
    assert rc == -1 and b"marlpde_rk45_stream_integrate_events_dev" in _cabi.lib().marlpde_last_error()
    assert _cabi.lib().marlpde_rk45_stream_workspace_bytes(64, 20000) > 9 * 64 * 5 * 20000 * 8
    assert _cabi.lib().marlpde_radau_workspace_bytes(1, 200) == 8 * 200 * (90 + 76 + 64)


def central_difference_jacobian(y, p):
    """Dense d rhs / d y of the oracle RHS by central differences (field-major), relative step 1e-7."""
    n = y.size
    J = np.zeros((n, n))
    fp, fm = np.empty(n), np.empty(n)
    for j in range(n):
        h = 1e-7 * max(1e-3, abs(y[j]))
        yp, ym = y.copy(), y.copy()
        yp[j] += h
        ym[j] -= h
        oracle.rhs(yp, p, fp)
        oracle.rhs(ym, p, fm)
        J[:, j] = (fp - fm) / (2 * h)
    return J


JAC_CASES = [("scenario_A", {"Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}, 5), ("high_porosity", {}, 13),
             ("high_porosity", {"time_varying_dPhi": True}, 9)]


@pytest.mark.parametrize("name,over,snap", JAC_CASES)
def test_analytic_jacobian_blocks(fixtures_reference, name, over, snap):
    """The implicit kernels write all three 5x5 Jacobian blocks of a cell analytically (csrc/implicit_common.cuh
    jac_analytic).  The formulas, restated in numpy (oracle/jacobian_blocks.py), against central differences of the
    oracle RHS on evolved states of the reference's own fixtures (all 200 cells, both column ends, the plain model and
    the time-varying-dPhi variant): off-diagonal blocks to 1e-8 of the largest Jacobian entry (the RHS is linear in
    the neighbour values), diagonal blocks to the accuracy of the difference quotient, and nothing outside the
    block-tridiagonal structure."""
    import jacobian_blocks as jb
    pde = oracle.derive_scenario({**oracle.default_scenario(), **over})
    p, N = oracle.kernel_params(pde), 200
    y = np.ascontiguousarray(fixtures_reference[name][snap], dtype=np.float64).reshape(-1)
    J = central_difference_jacobian(y, p)
    scale = np.abs(J).max()
    cells = np.arange(5 * N) % N
    assert np.abs(J[np.abs(cells[:, None] - cells[None, :]) > 1]).max() == 0.0
    for i in range(N):
        L, D, Ub = jb.blocks(y, p, i, N)
        rows = [f * N + i for f in range(5)]
        if i > 0:
            assert np.abs(J[np.ix_(rows, [f * N + i - 1 for f in range(5)])] - L).max() <= 1e-8 * scale
        if i < N - 1:
            assert np.abs(J[np.ix_(rows, [f * N + i + 1 for f in range(5)])] - Ub).max() <= 1e-8 * scale
        Jd = J[np.ix_(rows, rows)]
        assert np.all(np.abs(Jd - D) <= 1e-3 * np.abs(Jd) + 1e-9 * scale), (i, np.abs(Jd - D).max())


@pytest.mark.parametrize("n_cells", [1, 2, 3, 4, 5, 37, 200])
def test_two_ended_block_thomas_against_dense_solve(n_cells):
    """The linear algebra of the Radau kernel (csrc/radau_batch.cu factorise / solve: cells 0 .. N/2-1 eliminated
    top-down, N-1 .. N/2+1 bottom-up, meeting cell N/2; both chains of a solve in lock-step), restated in numpy
    (oracle/twisted_block_thomas.py), against a dense solve — for the real and the complex shift of scipy's Radau
    on the block-tridiagonal finite-difference Jacobian of the oracle RHS, and on random blocks for the tiny grids."""
    import twisted_block_thomas as tw
    rng = np.random.default_rng(n_cells)
    if n_cells >= 37:
        pde = oracle.default_scenario() | {"N": n_cells, "Phi0": 0.6, "PhiIni": 0.5, "PhiNR": 0.6}
        po = oracle.kernel_params(pde)
        y = (mb.initial_state(pde)[0] * (1 + 0.05 * rng.uniform(-1, 1, (5, n_cells)))).ravel()
        n = 5 * n_cells
        f0 = oracle.rhs(y, po, np.empty(n)).copy()
        Jf = np.empty((n, n))
        for j in range(n):
            d = 1e-7 * max(1e-3, abs(y[j]))
            yp = y.copy()
            yp[j] += d
            Jf[:, j] = (oracle.rhs(yp, po, np.empty(n)) - f0) / d
        perm = np.arange(n).reshape(5, n_cells).T.ravel()           # field-major -> cell-major
        Jc = Jf[np.ix_(perm, perm)]
        blk = lambda i, k: Jc[5 * i:5 * i + 5, 5 * k:5 * k + 5]
        D = np.stack([blk(i, i) for i in range(n_cells)])
        L = np.stack([blk(i, i - 1) if i > 0 else np.zeros((5, 5)) for i in range(n_cells)])
        U = np.stack([blk(i, i + 1) if i < n_cells - 1 else np.zeros((5, 5)) for i in range(n_cells)])
        # the Jacobian IS block tridiagonal in cell-major order (SURVEY.md 8a)
        T = np.zeros_like(Jc)
        for i in range(n_cells):
            for k in (i - 1, i, i + 1):
                if 0 <= k < n_cells:
                    T[5 * i:5 * i + 5, 5 * k:5 * k + 5] = blk(i, k)
        assert np.max(np.abs(Jc - T)) <= 1e-6 * np.max(np.abs(Jc))
        h = 1e-4
    else:
        D = rng.normal(size=(n_cells, 5, 5))
        L = 0.3 * rng.normal(size=(n_cells, 5, 5))
        U = 0.3 * rng.normal(size=(n_cells, 5, 5))
        h = 0.05
    for M in (3.637834252744496 / h, complex(2.6810828736277523, -3.050430199247411) / h):   # radau.py MU_REAL, MU_COMPLEX
        rhs = rng.normal(size=5 * n_cells)
        x = tw.solve(L, U, tw.factor(L, D, U, M), rhs)
        ref = np.linalg.solve(tw.dense(L, D, U, M), rhs)
        assert np.max(np.abs(x - ref)) <= 1e-11 * np.max(np.abs(ref))


def test_table_driven_fp64_maths_model_against_mpmath():
    """Tables (csrc/fp64_tables.inc), constants and algorithms of csrc/fp64_math.cuh, evaluated by an exact-FMA CPU
    model (oracle/fp64_math_model.py), against mpmath — same ranges and bounds as tests/test_gpu_math.py."""
    mp = pytest.importorskip("mpmath")
    import fp64_math_model as fm
    mp.mp.prec = 120
    c = fm.Constants(False)
    rng = np.random.default_rng(5)
    xs = np.concatenate([rng.uniform(1e-3, 3.0, 300), 10.0 ** rng.uniform(-300, 300, 100), 1 + rng.uniform(-1e-3, 1e-3, 100),
                         [1.0, 0.5, 2.0, np.nextafter(1, 0), np.nextafter(1, 2), 0.8, 0.6]])
    err = max(abs(mp.mpf(fm.log(c, float(x))) - mp.log(mp.mpf(float(x)))) / max(1, abs(mp.log(mp.mpf(float(x))))) for x in xs)
    assert err <= 2.5e-16
    xe = np.concatenate([rng.uniform(-40, 40, 300), rng.uniform(-689, 689, 100), rng.uniform(-1, 1, 100), [0.0]])
    err = max(abs(mp.mpf(fm.exp(c, float(x))) / mp.exp(mp.mpf(float(x))) - 1) for x in xe)
    assert err <= 4e-16
    xm = np.concatenate([rng.uniform(-200, 200, 200), rng.uniform(-1, 1, 200), rng.uniform(-0.03, 0.03, 200)])
    xm = xm[np.abs(xm) >= 1e-3]
    err = max(abs(mp.mpf(fm.expm1(c, float(x))) / mp.expm1(mp.mpf(float(x))) - 1) for x in xm)
    assert err <= 6e-16
    assert fm.exp(c, 0.0) == 1.0 and fm.log(c, 1.0) == 0.0

