"""Batched entry points over the C ABI: one RHS call, or a whole adaptive RK45 integration,
for many sediment columns at once.

Two flavours per operation, chosen by the type of the state argument:
  * numpy arrays  -> host-pointer ABI calls (`marlpde_rhs_batch`, `marlpde_rk45_integrate`):
                     the library copies H2D, runs the kernels, copies D2H.  This is the path the
                     reference-facing drop-in (`marlpde.integrate_equations`) and `bench.py`'s
                     `e2e` number use.
  * torch CUDA tensors -> device-pointer ABI calls (`*_dev`) on torch's current stream, with no
                     allocation or synchronisation inside the library (sweeps that keep their
                     columns resident in HBM, multi-GPU shards).
PyTorch is only plumbing here (device memory, streams); all arithmetic is in csrc/.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _cabi
from ._cabi import PARAMS_DTYPE, STATE_DTYPE, NEVENTS


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _as_params(params) -> np.ndarray:
    p = np.ascontiguousarray(params)
    if p.dtype != PARAMS_DTYPE:
        raise TypeError("params must come from marlpde_b200.derive_column_params")
    return p.reshape(-1)


def _check_y(y, n_columns):
    if y.ndim != 3 or y.shape[0] != n_columns or y.shape[1] != 5:
        raise ValueError(f"state must have shape (n_columns={n_columns}, 5, n_cells); got {tuple(y.shape)}")


def params_to_device(params, device):
    """Upload a params record array once (returns a uint8 CUDA tensor to pass back in)."""
    import torch
    p = _as_params(params)
    return torch.from_numpy(p.view(np.uint8).copy()).to(device)


def _model_flags(params) -> int:
    """MARLPDE_FLAG_* bits the integrators need for the model variants present in `params` (numpy records or the
    uint8 CUDA tensor of params_to_device): MARLPDE_FLAG_VAR_DPHI when any column carries MARLPDE_MODEL_VAR_DPHI."""
    off = PARAMS_DTYPE.fields["model_flags"][1]
    if _is_torch(params):
        import torch
        words = params.view(-1, PARAMS_DTYPE.itemsize)[:, off:off + 4].contiguous().view(torch.int32)
        any_var = bool((words & _cabi.MODEL_VAR_DPHI).any().item())
    else:
        any_var = bool(np.any(_as_params(params)["model_flags"] & _cabi.MODEL_VAR_DPHI))
    return _cabi.FLAG_VAR_DPHI if any_var else 0


def rhs_batch(y, params, out=None, device: int = 0):
    """dy/dt for every column: y[B,5,N] -> out[B,5,N] (replaces fun_numba/pde_rhs per column,
    marlpde/LHeureux_model.py:290-522)."""
    lib = _cabi.lib()
    if _is_torch(y):
        import torch
        if not y.is_cuda or y.dtype != torch.float64 or not y.is_contiguous():
            raise ValueError("device path needs a contiguous float64 CUDA tensor")
        d_params = params if _is_torch(params) else params_to_device(params, y.device)
        B = d_params.numel() // PARAMS_DTYPE.itemsize
        _check_y(y, B)
        if out is None:
            out = torch.empty_like(y)
        with torch.cuda.device(y.device):
            stream = torch.cuda.current_stream().cuda_stream
            _cabi.check(lib.marlpde_rhs_batch_dev(y.data_ptr(), d_params.data_ptr(), B, y.shape[2],
                                                  out.data_ptr(), stream))
        return out
    p = _as_params(params)
    y = np.ascontiguousarray(y, dtype=np.float64)
    _check_y(y, p.shape[0])
    if out is None:
        out = np.empty_like(y)
    _cabi.check(lib.marlpde_rhs_batch(_cabi.ptr(y), _cabi.ptr(p), p.shape[0], y.shape[2], _cabi.ptr(out), device))
    return out


@dataclass
class RK45Result:
    """Per-column results, the batched analogue of solve_ivp's OdeResult."""
    y: object                    # [B,5,N] state at the time reached
    t: np.ndarray                # [B] time reached
    h_abs: np.ndarray            # [B] next step size the controller would use
    status: np.ndarray           # [B] 0 finished, -1 step too small, 1 (2: mid-step, streaming path) step budget
                                 #     exhausted, resumable
    n_accepted: np.ndarray
    n_rejected: np.ndarray
    nfev: np.ndarray
    t_eval: np.ndarray           # [n_eval]
    snapshots: object            # [B,n_eval,5,N] dense-output samples (rows < next_eval are valid)
    next_eval: np.ndarray        # [B]
    event_counts: np.ndarray = None   # [B,7]
    event_times: np.ndarray = None    # [B,7,capacity]
    state: np.ndarray = field(default=None, repr=False)  # raw marlpde_column_state records (for resuming)

    @property
    def n_attempts(self):
        return self.n_accepted + self.n_rejected

    def solutions(self, column: int) -> np.ndarray:
        """(5, N, n_t) like `sol.y.reshape(5, N, -1)` in Evolve_scenario.py:168."""
        snap = self.snapshots[column]
        snap = snap.cpu().numpy() if _is_torch(snap) else np.asarray(snap)
        return np.ascontiguousarray(np.transpose(snap[: int(self.next_eval[column])], (1, 2, 0)))


def make_state(n_columns: int, t0=0.0, first_step=1e-6) -> np.ndarray:
    st = np.zeros(n_columns, dtype=STATE_DTYPE)
    st["t"] = t0
    st["h_abs"] = first_step
    return st


def integrate_rk45_batch(y0, params, t_span=(0.0, 1.0), first_step=1e-6, rtol=1e-3, atol=1e-3,
                         t_eval=None, max_step=np.inf, max_steps: int = 0, events: bool = False,
                         event_capacity: int = 0, state: np.ndarray | None = None,
                         device: int = 0, inplace: bool = False, quantum: int = 0) -> RK45Result:
    """Adaptive Dormand-Prince RK45 for every column, SciPy `solve_ivp(method="RK45")` semantics
    per column (call site marlpde/Evolve_scenario.py:104-109).

    `first_step` follows SciPy's rule (validate_first_step): it is used verbatim and must be
    positive and not exceed the interval.  `max_steps` > 0 bounds the step attempts per column in
    this call; columns that hit it come back with status 1 and can be resumed by passing the
    returned `.state` and `.y` back in.  `quantum` (on-chip kernel, `max_steps` > 0 only): step attempts per work
    item of the kernel's queue; 0 lets the library choose, a negative value claims whole columns.
    """
    lib = _cabi.lib()
    t0, t_bound = float(t_span[0]), float(t_span[1])
    if not t_bound > t0:
        raise ValueError("only forward integration (t_span[1] > t_span[0]) is supported")
    if state is None:
        fs = np.asarray(first_step, dtype=np.float64)
        if np.any(fs <= 0):
            raise ValueError("`first_step` must be positive.")
        if np.any(fs > abs(t_bound - t0)):
            raise ValueError("`first_step` exceeds bounds.")
    t_eval_arr = np.zeros(0) if t_eval is None else np.ascontiguousarray(t_eval, dtype=np.float64)
    if t_eval_arr.ndim != 1:
        raise ValueError("`t_eval` must be 1-dimensional.")
    if t_eval_arr.size:
        if np.any(t_eval_arr < t0) or np.any(t_eval_arr > t_bound):
            raise ValueError("Values in `t_eval` are not within `t_span`.")
        if np.any(np.diff(t_eval_arr) <= 0):
            raise ValueError("Values in `t_eval` are not properly sorted.")
    n_eval = int(t_eval_arr.size)
    cap = int(event_capacity) if events else 0
    opts = _cabi.RK45Options(t_bound=t_bound, rtol=float(rtol), atol=float(atol), max_step=float(max_step),
                             max_steps=int(max_steps), n_eval=n_eval, event_capacity=cap,
                             flags=(_cabi.FLAG_EVENTS if events else 0) | _cabi.FLAG_QUEUE_LOCKS | _model_flags(params),
                             quantum=int(quantum))

    if _is_torch(y0):
        import torch
        if not y0.is_cuda or y0.dtype != torch.float64 or not y0.is_contiguous():
            raise ValueError("device path needs a contiguous float64 CUDA tensor")
        dev = y0.device
        d_params = params if _is_torch(params) else params_to_device(params, dev)
        B = d_params.numel() // PARAMS_DTYPE.itemsize
        _check_y(y0, B)
        N = y0.shape[2]
        st = make_state(B, t0, first_step) if state is None else np.ascontiguousarray(state, dtype=STATE_DTYPE)
        y = y0 if inplace else y0.clone()
        if B and (N > lib.marlpde_rk45_max_cells() or N < 32):
            return _stream_rk45_device(lib, y, d_params, st, opts, t_eval_arr, B, N, dev, cap)
        with torch.cuda.device(dev):
            d_state = torch.from_numpy(st.view(np.uint8).copy()).to(dev)
            d_te = torch.from_numpy(t_eval_arr.copy()).to(dev) if n_eval else None
            d_snap = torch.full((B, n_eval, 5, N), float("nan"), dtype=torch.float64, device=dev)   # rows >= next_eval stay NaN
            d_queue = torch.zeros(1 + 2 * B, dtype=torch.int32, device=dev)   # work counter + lock word and attempt counter per column
            d_ec = torch.zeros((B, NEVENTS), dtype=torch.int32, device=dev)
            d_et = torch.full((B, NEVENTS, max(cap, 1)), float("nan"), dtype=torch.float64, device=dev)
            stream = torch.cuda.current_stream().cuda_stream
            _cabi.check(lib.marlpde_rk45_integrate_dev(
                y.data_ptr(), d_params.data_ptr(), d_state.data_ptr(), B, N, C.byref(opts),
                d_te.data_ptr() if n_eval else None, d_snap.data_ptr(), d_ec.data_ptr(), d_et.data_ptr(),
                d_queue.data_ptr(), stream))
            st_out = d_state.cpu().numpy().view(STATE_DTYPE).reshape(B)   # synchronises the stream
            ec, et = d_ec.cpu().numpy(), d_et.cpu().numpy()[:, :, :cap]
        snaps = d_snap
    else:
        p = _as_params(params)
        B = p.shape[0]
        y = np.array(y0, dtype=np.float64, order="C", copy=not inplace)
        _check_y(y, B)
        N = y.shape[2]
        st_out = make_state(B, t0, first_step) if state is None else np.array(state, dtype=STATE_DTYPE, copy=True)
        snaps = np.full((B, n_eval, 5, N), np.nan)
        ec = np.zeros((B, NEVENTS), dtype=np.int32)
        et = np.full((B, NEVENTS, cap), np.nan)
        _cabi.check(lib.marlpde_rk45_integrate(
            _cabi.ptr(y), _cabi.ptr(p), _cabi.ptr(st_out), B, N, C.byref(opts),
            _cabi.ptr(t_eval_arr) if n_eval else None, _cabi.ptr(snaps) if n_eval else None,
            _cabi.ptr(ec), _cabi.ptr(et) if cap else None, device))
    return RK45Result(y=y, t=st_out["t"].copy(), h_abs=st_out["h_abs"].copy(), status=st_out["status"].copy(),
                      n_accepted=st_out["n_accepted"].copy(), n_rejected=st_out["n_rejected"].copy(),
                      nfev=st_out["nfev"].copy(), t_eval=t_eval_arr, snapshots=snaps,
                      next_eval=st_out["next_eval"].copy(), event_counts=ec, event_times=et, state=st_out)


def _stream_rk45_device(lib, y, d_params, st, opts, t_eval_arr, B, N, dev, cap, batch: int = 512):
    """Depth grids that do not fit on chip: repeat fixed-size batches of step attempts of the streaming
    kernels (csrc/rk45_streaming.cu) on torch's current stream until every column has finished or
    `max_steps` is used up.  The per-batch status read-back is the only host round trip."""
    import torch
    n_eval = int(t_eval_arr.size)
    budget = int(opts.max_steps)
    with torch.cuda.device(dev):
        d_state = torch.from_numpy(st.view(np.uint8).copy()).to(dev)
        d_te = torch.from_numpy(t_eval_arr.copy()).to(dev) if n_eval else None
        d_snap = torch.full((B, n_eval, 5, N), float("nan"), dtype=torch.float64, device=dev)   # rows >= next_eval stay NaN
        nb = int(lib.marlpde_rk45_stream_workspace_bytes(B, N))
        d_work = torch.empty(nb // 8 + 1, dtype=torch.float64, device=dev)
        d_ec = torch.zeros((B, NEVENTS), dtype=torch.int32, device=dev)
        d_et = torch.full((B, NEVENTS, max(cap, 1)), float("nan"), dtype=torch.float64, device=dev)
        stream = torch.cuda.current_stream().cuda_stream
        used = 0
        while True:
            o = _cabi.RK45Options(t_bound=opts.t_bound, rtol=opts.rtol, atol=opts.atol, max_step=opts.max_step,
                                  max_steps=min(batch, budget - used) if budget > 0 else batch, n_eval=n_eval,
                                  event_capacity=opts.event_capacity, flags=opts.flags, quantum=0)
            _cabi.check(lib.marlpde_rk45_stream_integrate_events_dev(
                y.data_ptr(), d_params.data_ptr(), d_state.data_ptr(), B, N, C.byref(o),
                d_te.data_ptr() if n_eval else None, d_snap.data_ptr(), d_ec.data_ptr(), d_et.data_ptr(),
                d_work.data_ptr(), nb, stream))
            used += int(o.max_steps)
            st_out = d_state.cpu().numpy().view(STATE_DTYPE).reshape(B)
            if not np.any(st_out["status"] >= 1) or (budget > 0 and used >= budget):
                break
            d_state = torch.from_numpy(st_out.view(np.uint8).copy()).to(dev)
        ec, et = d_ec.cpu().numpy(), d_et.cpu().numpy()[:, :, :cap]
    return RK45Result(y=y, t=st_out["t"].copy(), h_abs=st_out["h_abs"].copy(), status=st_out["status"].copy(),
                      n_accepted=st_out["n_accepted"].copy(), n_rejected=st_out["n_rejected"].copy(),
                      nfev=st_out["nfev"].copy(), t_eval=t_eval_arr, snapshots=d_snap,
                      next_eval=st_out["next_eval"].copy(), event_counts=ec, event_times=et, state=st_out)


@dataclass
class RadauResult:
    """Per-column results of the implicit integrator (batched analogue of solve_ivp's OdeResult)."""
    y: object                    # [B,5,N] state at the time reached
    t: np.ndarray                # [B]
    h_abs: np.ndarray            # [B] next step size
    status: np.ndarray           # [B] 0 finished, -1 step too small, 1 step budget exhausted
    n_accepted: np.ndarray       # accepted steps
    n_rejected: np.ndarray       # steps rejected by the error test
    nfev: np.ndarray
    njev: np.ndarray             # Jacobians (analytic off-diagonal blocks + 5 RHS evaluations each, counted in nfev)
    nlu: np.ndarray              # block-tridiagonal factorisations (real and complex counted separately)
    newton_iterations: np.ndarray
    newton_failures: np.ndarray
    t_eval: np.ndarray
    snapshots: object            # [B,n_eval,5,N]
    next_eval: np.ndarray
    event_counts: np.ndarray = None   # [B,7]
    event_times: np.ndarray = None    # [B,7,capacity]
    state: np.ndarray = field(default=None, repr=False)
    # forward sensitivities (integrate_bdf_batch(..., sensitivities=...)); None without them
    sensitivities: object = None      # [B,P,n_eval,5,N] s = dy/d eps at t_eval (rows < next_eval are valid)
    sens_y: object = None             # [B,P,5,N] s at the time reached (the w of a resumed call)
    sens_stats: np.ndarray = None     # [B,3] corrector iterations, fallback factorisations, unconverged steps

    def solutions(self, column: int) -> np.ndarray:
        snap = self.snapshots[column]
        snap = snap.cpu().numpy() if _is_torch(snap) else np.asarray(snap)
        return np.ascontiguousarray(np.transpose(snap[: int(self.next_eval[column])], (1, 2, 0)))

    @property
    def work(self) -> np.ndarray:
        """Relative cost each column turned out to have (step attempts incl. failed Newton episodes).  Columns are
        claimed from a queue in batch order and a column is sequential in time, so a sweep that is repeated (other
        t_eval, a neighbouring parameter set) finishes sooner when the columns are passed longest-first:
        `order = np.argsort(-previous.work)` — or, a priori, `np.argsort(-sweep.predicted_cost(pde, "Radau"))`
        (4096-column lattice to T*: 21.2 s in lattice order, 18.3 s by the estimate, 17.9-18.5 s by measured work)."""
        return self.n_accepted + self.n_rejected + self.newton_failures


def integrate_radau_batch(y0, params, t_span=(0.0, 1.0), first_step=1e-6, rtol=1e-3, atol=1e-3, t_eval=None,
                          max_step=np.inf, max_steps: int = 0, events: bool = False, event_capacity: int = 0,
                          state: np.ndarray | None = None, device: int = 0, inplace: bool = False,
                          jac: str = "analytic", team_columns="auto") -> RadauResult:
    """Implicit integration of every column: 3-stage Radau IIA with SciPy's step-size, Newton and
    Jacobian-reuse rules (`solve_ivp(method="Radau", jac_sparsity=jacobian_sparsity())`, the
    reference's default Solver, parameters.py:201-221) and a block-tridiagonal linear solver.
    `team_columns`: the first K columns of the batch are integrated by two warps each (the latency shape: ~1.4x faster
    per column at twice the slots) — "auto": every column of a batch that leaves the GPU half empty anyway (<= 296
    columns), none otherwise; a sweep passes its longest columns first and a K (sweep.team_columns)."""
    return _integrate_implicit("radau", y0, params, t_span, first_step, rtol, atol, t_eval, max_step, max_steps, events,
                               event_capacity, state, device, inplace, jac, team_columns)


def integrate_bdf_batch(y0, params, t_span=(0.0, 1.0), first_step=1e-6, rtol=1e-3, atol=1e-3, t_eval=None,
                        max_step=np.inf, max_steps: int = 0, events: bool = False, event_capacity: int = 0,
                        state: np.ndarray | None = None, device: int = 0, inplace: bool = False,
                          jac: str = "analytic", sensitivities=None, sens_y=None, sens_atol=None) -> RadauResult:
    """Implicit integration of every column with the variable-order BDF kernel (csrc/bdf_batch.cu): SciPy's `BDF`
    step for step (`solve_ivp(method="BDF", jac_sparsity=jacobian_sparsity())`, parameters.py:235-236) on the
    block-tridiagonal linear solver of the Radau kernel; also what `method="LSODA"` batches run on the device
    (parameters.py:214-219: LSODA is a BDF code on this stiff system).  Same result type as the Radau path; `nlu`
    counts one real factorisation each.  A column resumed from `state` restarts at order 1.

    `sensitivities` (a `marlpde_b200.sensitivity_directions(pde, wrt)` object for the same columns) adds forward
    parameter sensitivities s_k = dy/d eps_k along each direction (staggered direct method, excluded from the error
    control, DESIGN.md 5.4): the state's path is bit-identical to a run without them.  Derivatives are taken at fixed
    nondimensional time t (a direction that moves Tstar gives dy(t)/d eps at fixed t, not at fixed years).  The result
    then carries `sensitivities` [B,P,n_eval,5,N], `sens_y` [B,P,5,N] (s at the time reached) and `sens_stats` [B,3].
    `sens_y` (default: the directions' w = dy0/d eps) is s at the start time — pass a budget-stopped result's `.sens_y`
    back with its `.state` to resume; `sens_atol` [B,P] (default `sensitivities.atol(atol)`) is the absolute tolerance
    of s in the corrector's convergence test."""
    sens = None
    if sensitivities is not None:
        sens = (sensitivities, sensitivities.w if sens_y is None else sens_y,
                sensitivities.atol(atol) if sens_atol is None else sens_atol)
    return _integrate_implicit("bdf", y0, params, t_span, first_step, rtol, atol, t_eval, max_step, max_steps, events,
                               event_capacity, state, device, inplace, jac, sens=sens)


TEAM_AUTO_MAX_COLUMNS = 296     # 2 per SM: below this every column gets a two-warp team ("auto")


def _integrate_implicit(kind, y0, params, t_span, first_step, rtol, atol, t_eval, max_step, max_steps, events,
                        event_capacity, state, device, inplace, jac="analytic", team_columns=0, sens=None) -> RadauResult:
    """`jac`: "analytic" (default) — every 5x5 block analytic in one pass, no RHS evaluations; only for a cell that sits ON
    a switching surface of the model the porosity column is num_jac's one-sided difference (csrc/implicit_common.cuh);
    "fd" (MARLPDE_FLAG_JAC_FD) — analytic off-diagonal blocks, diagonal blocks by finite differences with num_jac's step
    rule everywhere (what SciPy forms; 5 RHS evaluations per Jacobian, ~9 % slower, same robustness)."""
    if jac not in ("fd", "analytic"):
        raise ValueError("jac must be 'fd' or 'analytic'")
    lib = _cabi.lib()
    f_ws = getattr(lib, f"marlpde_{kind}_workspace_bytes")
    f_dev = getattr(lib, f"marlpde_{kind}_integrate_dev")
    f_host = getattr(lib, f"marlpde_{kind}_integrate")
    t0, t_bound = float(t_span[0]), float(t_span[1])
    if not t_bound > t0:
        raise ValueError("only forward integration (t_span[1] > t_span[0]) is supported")
    if state is None:
        fs = np.asarray(first_step, dtype=np.float64)
        if np.any(fs <= 0):
            raise ValueError("`first_step` must be positive.")
        if np.any(fs > abs(t_bound - t0)):
            raise ValueError("`first_step` exceeds bounds.")
    t_eval_arr = np.zeros(0) if t_eval is None else np.ascontiguousarray(t_eval, dtype=np.float64)
    if t_eval_arr.ndim != 1:
        raise ValueError("`t_eval` must be 1-dimensional.")
    if t_eval_arr.size:
        if np.any(t_eval_arr < t0) or np.any(t_eval_arr > t_bound):
            raise ValueError("Values in `t_eval` are not within `t_span`.")
        if np.any(np.diff(t_eval_arr) <= 0):
            raise ValueError("Values in `t_eval` are not properly sorted.")
    n_eval = int(t_eval_arr.size)
    cap = int(event_capacity) if events else 0
    opts = _cabi.RK45Options(t_bound=t_bound, rtol=float(rtol), atol=float(atol), max_step=float(max_step),
                             max_steps=int(max_steps), n_eval=n_eval, event_capacity=cap,
                             flags=(_cabi.FLAG_EVENTS if events else 0) | _model_flags(params)
                             | (_cabi.FLAG_JAC_FD if jac == "fd" else 0), quantum=0)
    n_batch = int(y0.shape[0])
    if kind != "radau" or jac == "fd":
        team = 0
    elif team_columns == "auto":
        team = n_batch if n_batch <= TEAM_AUTO_MAX_COLUMNS else 0
    else:
        team = max(0, min(int(team_columns), n_batch))
    opts.quantum = team
    if _is_torch(y0):
        import torch
        if not y0.is_cuda or y0.dtype != torch.float64 or not y0.is_contiguous():
            raise ValueError("device path needs a contiguous float64 CUDA tensor")
        dev = y0.device
        d_params = params if _is_torch(params) else params_to_device(params, dev)
        B = d_params.numel() // PARAMS_DTYPE.itemsize
        _check_y(y0, B)
        N = y0.shape[2]
        st = make_state(B, t0, first_step) if state is None else np.ascontiguousarray(state, dtype=STATE_DTYPE)
        y = y0 if inplace else y0.clone()
        with torch.cuda.device(dev):
            d_state = torch.from_numpy(st.view(np.uint8).copy()).to(dev)
            d_te = torch.from_numpy(t_eval_arr.copy()).to(dev) if n_eval else None
            d_snap = torch.full((B, n_eval, 5, N), float("nan"), dtype=torch.float64, device=dev)   # rows >= next_eval stay NaN
            d_queue = torch.zeros(2, dtype=torch.int32, device=dev)     # [1]: the team launch's queue
            d_stats = torch.zeros((B, 4), dtype=torch.int64, device=dev)
            d_ec = torch.zeros((B, NEVENTS), dtype=torch.int32, device=dev)
            d_et = torch.full((B, NEVENTS, max(cap, 1)), float("nan"), dtype=torch.float64, device=dev)
            nb = int(f_ws(B, N))
            d_work = torch.empty(max(nb, 8) // 8, dtype=torch.float64, device=dev)
            stream = torch.cuda.current_stream().cuda_stream
            if sens is None:
                _cabi.check(f_dev(
                    y.data_ptr(), d_params.data_ptr(), d_state.data_ptr(), B, N, C.byref(opts),
                    d_te.data_ptr() if n_eval else None, d_snap.data_ptr(), d_ec.data_ptr(), d_et.data_ptr(),
                    d_stats.data_ptr(), d_work.data_ptr(), nb, d_queue.data_ptr(), stream))
            else:
                sd, sy, sat = _sens_inputs(sens, B, N)
                P = sd.n_dirs
                d_pm = torch.from_numpy(sd.params_pm.view(np.uint8).reshape(-1).copy()).to(dev)
                d_i2s = torch.from_numpy(sd.inv2sigma.copy()).to(dev)
                d_sat = torch.from_numpy(sat.copy()).to(dev)
                d_sens = (sy.clone() if _is_torch(sy) else torch.from_numpy(np.array(sy)).to(dev)).contiguous()
                d_ssnap = torch.full((B, P, n_eval, 5, N), float("nan"), dtype=torch.float64, device=dev)
                d_sstats = torch.zeros((B, 3), dtype=torch.int64, device=dev)
                nbs = int(lib.marlpde_bdf_sens_workspace_bytes(B, N, P))
                d_swork = torch.empty(max(nbs, 8) // 8, dtype=torch.float64, device=dev)
                _cabi.check(lib.marlpde_bdf_sens_integrate_dev(
                    y.data_ptr(), d_params.data_ptr(), d_state.data_ptr(), B, N, C.byref(opts),
                    d_te.data_ptr() if n_eval else None, d_snap.data_ptr(), d_ec.data_ptr(), d_et.data_ptr(),
                    d_stats.data_ptr(), d_work.data_ptr(), nb, d_queue.data_ptr(), P, d_pm.data_ptr(),
                    d_i2s.data_ptr(), d_sat.data_ptr(), d_sens.data_ptr(), d_ssnap.data_ptr(), d_sstats.data_ptr(),
                    d_swork.data_ptr(), nbs, stream))
                sens_out = (d_ssnap, d_sens, d_sstats.cpu().numpy())
            st_out = d_state.cpu().numpy().view(STATE_DTYPE).reshape(B)
            stats = d_stats.cpu().numpy()
            ec, et = d_ec.cpu().numpy(), d_et.cpu().numpy()[:, :, :cap]
        snaps = d_snap
    else:
        p = _as_params(params)
        B = p.shape[0]
        y = np.array(y0, dtype=np.float64, order="C", copy=not inplace)
        _check_y(y, B)
        N = y.shape[2]
        st_out = make_state(B, t0, first_step) if state is None else np.array(state, dtype=STATE_DTYPE, copy=True)
        snaps = np.full((B, n_eval, 5, N), np.nan)
        stats = np.zeros((B, 4), dtype=np.int64)
        ec = np.zeros((B, NEVENTS), dtype=np.int32)
        et = np.full((B, NEVENTS, cap), np.nan)
        if sens is None:
            _cabi.check(f_host(
                _cabi.ptr(y), _cabi.ptr(p), _cabi.ptr(st_out), B, N, C.byref(opts),
                _cabi.ptr(t_eval_arr) if n_eval else None, _cabi.ptr(snaps) if n_eval else None, _cabi.ptr(ec),
                _cabi.ptr(et) if cap else None, _cabi.ptr(stats), device))
        else:
            sd, sy, sat = _sens_inputs(sens, B, N)
            P = sd.n_dirs
            s_y = np.array(sy.cpu().numpy() if _is_torch(sy) else sy, dtype=np.float64, order="C", copy=True)
            s_snap = np.full((B, P, n_eval, 5, N), np.nan)
            s_stats = np.zeros((B, 3), dtype=np.int64)
            _cabi.check(lib.marlpde_bdf_sens_integrate(
                _cabi.ptr(y), _cabi.ptr(p), _cabi.ptr(st_out), B, N, C.byref(opts),
                _cabi.ptr(t_eval_arr) if n_eval else None, _cabi.ptr(snaps) if n_eval else None, _cabi.ptr(ec),
                _cabi.ptr(et) if cap else None, _cabi.ptr(stats), P, _cabi.ptr(sd.params_pm), _cabi.ptr(sd.inv2sigma),
                _cabi.ptr(sat), _cabi.ptr(s_y), _cabi.ptr(s_snap) if n_eval else None, _cabi.ptr(s_stats), device))
            sens_out = (s_snap, s_y, s_stats)
    extra = {} if sens is None else dict(sensitivities=sens_out[0], sens_y=sens_out[1], sens_stats=sens_out[2])
    return RadauResult(y=y, t=st_out["t"].copy(), h_abs=st_out["h_abs"].copy(), status=st_out["status"].copy(),
                       n_accepted=st_out["n_accepted"].copy(), n_rejected=st_out["n_rejected"].copy(),
                       nfev=st_out["nfev"].copy(), njev=stats[:, 0].copy(), nlu=stats[:, 1].copy(),
                       newton_iterations=stats[:, 2].copy(), newton_failures=stats[:, 3].copy(),
                       t_eval=t_eval_arr, snapshots=snaps, next_eval=st_out["next_eval"].copy(), event_counts=ec,
                       event_times=et, state=st_out, **extra)


def _sens_inputs(sens, B, N):
    """Checked (directions, s at the start time [B,P,5,N], atol_s [B,P]) of a sensitivity run."""
    sd, sy, sat = sens
    P = sd.n_dirs
    if sd.params_pm.shape != (B, P, 2) or sd.w.shape != (B, P, 5, N):
        raise ValueError(f"sensitivity directions were derived for {sd.params_pm.shape[0]} columns of "
                         f"{sd.w.shape[-1]} cells, the batch has {B} of {N}")
    if tuple(sy.shape) != (B, P, 5, N):
        raise ValueError(f"sens_y must have shape {(B, P, 5, N)}; got {tuple(sy.shape)}")
    sat = np.ascontiguousarray(np.broadcast_to(np.asarray(sat, dtype=np.float64), (B, P)))
    if np.any(~(sat > 0)):
        raise ValueError("sens_atol must be positive")
    return sd, sy, sat


def integrate_rk23_batch(y0, params, t_span=(0.0, 1.0), first_step=1e-6, rtol=1e-3, atol=1e-3, t_eval=None,
                         max_step=np.inf, max_steps: int = 0, events: bool = False, event_capacity: int = 0,
                         state: np.ndarray | None = None, device: int = 0, inplace: bool = False) -> RK45Result:
    """Adaptive Bogacki-Shampine RK23 for every column (csrc/erk_batch.cu), SciPy `solve_ivp(method="RK23")` semantics
    per column: same step-size control and error norm, cubic dense output for `t_eval` and event location.  Arguments
    and result as for `integrate_rk45_batch` (no `quantum`); a column that stops on `max_steps` stops after an accepted
    step and resumes from the returned `.state` and `.y` exactly as if it had not stopped."""
    return _integrate_erk("rk23", y0, params, t_span, first_step, rtol, atol, t_eval, max_step, max_steps, events,
                          event_capacity, state, device, inplace)


def integrate_dop853_batch(y0, params, t_span=(0.0, 1.0), first_step=1e-6, rtol=1e-3, atol=1e-3, t_eval=None,
                           max_step=np.inf, max_steps: int = 0, events: bool = False, event_capacity: int = 0,
                           state: np.ndarray | None = None, device: int = 0, inplace: bool = False) -> RK45Result:
    """Adaptive Dormand-Prince DOP853 for every column (csrc/erk_batch.cu), SciPy `solve_ivp(method="DOP853")`
    semantics per column, including the seventh-order dense output whose three extra RHS evaluations are spent (and
    counted in `nfev`) only in steps that sample `t_eval` or locate an event.  Arguments and result as for
    `integrate_rk23_batch`."""
    return _integrate_erk("dop853", y0, params, t_span, first_step, rtol, atol, t_eval, max_step, max_steps, events,
                          event_capacity, state, device, inplace)


def _integrate_erk(kind, y0, params, t_span, first_step, rtol, atol, t_eval, max_step, max_steps, events,
                   event_capacity, state, device, inplace) -> RK45Result:
    lib = _cabi.lib()
    f_ws = getattr(lib, f"marlpde_{kind}_workspace_bytes")
    f_dev = getattr(lib, f"marlpde_{kind}_integrate_dev")
    f_host = getattr(lib, f"marlpde_{kind}_integrate")
    t0, t_bound = float(t_span[0]), float(t_span[1])
    if not t_bound > t0:
        raise ValueError("only forward integration (t_span[1] > t_span[0]) is supported")
    if state is None:
        fs = np.asarray(first_step, dtype=np.float64)
        if np.any(fs <= 0):
            raise ValueError("`first_step` must be positive.")
        if np.any(fs > abs(t_bound - t0)):
            raise ValueError("`first_step` exceeds bounds.")
    t_eval_arr = np.zeros(0) if t_eval is None else np.ascontiguousarray(t_eval, dtype=np.float64)
    if t_eval_arr.ndim != 1:
        raise ValueError("`t_eval` must be 1-dimensional.")
    if t_eval_arr.size:
        if np.any(t_eval_arr < t0) or np.any(t_eval_arr > t_bound):
            raise ValueError("Values in `t_eval` are not within `t_span`.")
        if np.any(np.diff(t_eval_arr) <= 0):
            raise ValueError("Values in `t_eval` are not properly sorted.")
    n_eval = int(t_eval_arr.size)
    cap = int(event_capacity) if events else 0
    opts = _cabi.RK45Options(t_bound=t_bound, rtol=float(rtol), atol=float(atol), max_step=float(max_step),
                             max_steps=int(max_steps), n_eval=n_eval, event_capacity=cap,
                             flags=(_cabi.FLAG_EVENTS if events else 0) | _model_flags(params), quantum=0)
    if _is_torch(y0):
        import torch
        if not y0.is_cuda or y0.dtype != torch.float64 or not y0.is_contiguous():
            raise ValueError("device path needs a contiguous float64 CUDA tensor")
        dev = y0.device
        d_params = params if _is_torch(params) else params_to_device(params, dev)
        B = d_params.numel() // PARAMS_DTYPE.itemsize
        _check_y(y0, B)
        N = y0.shape[2]
        st = make_state(B, t0, first_step) if state is None else np.ascontiguousarray(state, dtype=STATE_DTYPE)
        y = y0 if inplace else y0.clone()
        with torch.cuda.device(dev):
            d_state = torch.from_numpy(st.view(np.uint8).copy()).to(dev)
            d_te = torch.from_numpy(t_eval_arr.copy()).to(dev) if n_eval else None
            d_snap = torch.full((B, n_eval, 5, N), float("nan"), dtype=torch.float64, device=dev)   # rows >= next_eval stay NaN
            d_queue = torch.zeros(1, dtype=torch.int32, device=dev)
            d_ec = torch.zeros((B, NEVENTS), dtype=torch.int32, device=dev)
            d_et = torch.full((B, NEVENTS, max(cap, 1)), float("nan"), dtype=torch.float64, device=dev)
            nb = int(f_ws(B, N))
            d_work = torch.empty(max(nb, 8) // 8, dtype=torch.float64, device=dev)
            stream = torch.cuda.current_stream().cuda_stream
            _cabi.check(f_dev(
                y.data_ptr(), d_params.data_ptr(), d_state.data_ptr(), B, N, C.byref(opts),
                d_te.data_ptr() if n_eval else None, d_snap.data_ptr(), d_ec.data_ptr(), d_et.data_ptr(),
                d_work.data_ptr(), nb, d_queue.data_ptr(), stream))
            st_out = d_state.cpu().numpy().view(STATE_DTYPE).reshape(B)   # synchronises the stream
            ec, et = d_ec.cpu().numpy(), d_et.cpu().numpy()[:, :, :cap]
        snaps = d_snap
    else:
        p = _as_params(params)
        B = p.shape[0]
        y = np.array(y0, dtype=np.float64, order="C", copy=not inplace)
        _check_y(y, B)
        N = y.shape[2]
        st_out = make_state(B, t0, first_step) if state is None else np.array(state, dtype=STATE_DTYPE, copy=True)
        snaps = np.full((B, n_eval, 5, N), np.nan)
        ec = np.zeros((B, NEVENTS), dtype=np.int32)
        et = np.full((B, NEVENTS, cap), np.nan)
        _cabi.check(f_host(
            _cabi.ptr(y), _cabi.ptr(p), _cabi.ptr(st_out), B, N, C.byref(opts),
            _cabi.ptr(t_eval_arr) if n_eval else None, _cabi.ptr(snaps) if n_eval else None,
            _cabi.ptr(ec), _cabi.ptr(et) if cap else None, device))
    return RK45Result(y=y, t=st_out["t"].copy(), h_abs=st_out["h_abs"].copy(), status=st_out["status"].copy(),
                      n_accepted=st_out["n_accepted"].copy(), n_rejected=st_out["n_rejected"].copy(),
                      nfev=st_out["nfev"].copy(), t_eval=t_eval_arr, snapshots=snaps,
                      next_eval=st_out["next_eval"].copy(), event_counts=ec, event_times=et, state=st_out)
