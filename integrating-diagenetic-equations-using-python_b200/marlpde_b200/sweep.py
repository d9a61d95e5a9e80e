"""Parameter sweeps over several GPUs: columns are independent, so they are sharded column-wise,
one process per GPU, with NO collective on the data path; the only exchange is one all-gather of
the results after the integration (SURVEY.md §8e, BASELINE.json configs[2]).

    partition / balanced_assignment   which rank integrates which column
    shard                             a rank's slice of a Map_Scenario sweep dictionary
    gather_columns                    the collective: per-rank [b_r, ...] arrays -> [B, ...] on every rank
    sweep_rk45 / sweep_radau          shard -> integrate_{rk45,radau}_batch on this rank's GPU -> gather

`torch.distributed` is plumbing only (NCCL over NVLink on GPUs; the tests drive the same code with
gloo on CPU tensors and a stand-in integrator).  The reference has no counterpart: it integrates
one column per process (marlpde/Evolve_scenario.py:19).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np


def partition(n_columns: int, world_size: int) -> list[tuple[int, int]]:
    """Contiguous column blocks, sizes differing by at most one: [(start, stop)] per rank."""
    if world_size < 1 or n_columns < 0:
        raise ValueError("need world_size >= 1 and n_columns >= 0")
    base, extra = divmod(n_columns, world_size)
    out, start = [], 0
    for r in range(world_size):
        stop = start + base + (1 if r < extra else 0)
        out.append((start, stop))
        start = stop
    return out


def predicted_cost(pde: dict, method: str = "RK45") -> np.ndarray:
    """Relative cost of integrating a column to T*, used only to ORDER columns (longest first) and to balance shards.

    RK45: number of explicit steps — the step size is bound by the diffusive stability limit,
    steps ~ rho(J) ~ dCO3 * (Xstar * N / max_depth)^2 (SURVEY.md §8d).
    Radau: the implicit integrator does not see that limit; its work (step attempts incl. failed Newton episodes) is
    governed by how sharp the porosity front gets, i.e. by the compaction coefficient b (dPhi ~ 1/b).  Empirical fit on
    the 4096-column benchmark lattice (default base, r02o): work ~ b^2.16 S^-0.66 DCO3^0.05, rank correlation 0.996 —
    the a-priori RK45 estimate has correlation 0.13 with it.
    RK23, DOP853: the explicit estimate of RK45 — every explicit method is held at its stability limit on this system —
    NOT fitted for these methods (their stability regions differ from RK45's only by a constant factor, which does not
    change the order)."""
    if method in ("Radau", "BDF"):    # (BDF: same front-sharpness dependence; not fitted separately)
        b = np.atleast_1d(np.asarray(pde["b"], dtype=np.float64))
        srate = np.atleast_1d(np.asarray(pde["sedimentationrate"], dtype=np.float64))
        cost = b ** 2.16 * srate ** -0.66
        return np.broadcast_to(cost, np.broadcast_shapes(np.shape(b), np.shape(srate))).astype(np.float64)
    n = int(pde["N"])
    xstar = np.atleast_1d(np.asarray(pde["Xstar"], dtype=np.float64))
    d = np.atleast_1d(np.asarray(pde["DCO3"], dtype=np.float64)) / np.asarray(pde["D0Ca"], dtype=np.float64)
    cost = d * (xstar * n / np.asarray(pde["max_depth"], dtype=np.float64)) ** 2
    return np.broadcast_to(cost, np.broadcast_shapes(np.shape(xstar), np.shape(d))).astype(np.float64)


def balanced_assignment(cost: np.ndarray, world_size: int) -> list[np.ndarray]:
    """Column indices per rank: columns sorted by predicted cost (descending, stable) are dealt out
    in a boustrophedon order (0..W-1, W-1..0, ...), so every rank gets the same count (+-1) and
    nearly the same total cost.  Deterministic: every rank computes the same assignment."""
    order = np.argsort(-np.asarray(cost, dtype=np.float64), kind="stable")
    ranks = [[] for _ in range(world_size)]
    for pos, c in enumerate(order):
        lap, r = divmod(pos, world_size)
        ranks[r if lap % 2 == 0 else world_size - 1 - r].append(int(c))
    return [np.asarray(sorted(r), dtype=np.int64) for r in ranks]


def n_columns_of(pde: dict) -> int:
    n = 1
    for k, v in pde.items():
        if k != "N" and np.ndim(v) == 1:
            n = max(n, len(v))
    return n


def shard(pde: dict, columns) -> dict:
    """The sweep dictionary restricted to `columns` (a slice or an index array); scalars stay scalars."""
    return {k: (np.asarray(v)[columns] if (k != "N" and np.ndim(v) == 1) else v) for k, v in pde.items()}


def gather_columns(local, counts, group=None):
    """All-gather of per-rank arrays whose first axis is the rank's column count.

    `local`: torch tensor [b_r, ...] (CUDA -> NCCL, CPU -> gloo); `counts`: column count of every rank.
    Shards are padded to max(counts) so one equal-size `all_gather_into_tensor` does it (the NCCL
    fast path), then the padding is dropped.  Returns [sum(counts), ...] in rank order."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return local
    if len(counts) != world:
        raise ValueError("counts must have one entry per rank")
    bmax = int(max(counts))
    pad = local
    if local.shape[0] != bmax:
        pad = torch.zeros((bmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        pad[: local.shape[0]] = local
    out = torch.empty((world * bmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, pad.contiguous(), group=group)
    if all(int(c) == bmax for c in counts):
        return out
    return torch.cat([out[r * bmax: r * bmax + int(c)] for r, c in enumerate(counts)], dim=0)


@dataclass
class SweepResult:
    """Results for ALL columns of the sweep, identical on every rank, in the original column order."""
    y: np.ndarray            # [B,5,N] end states
    snapshots: np.ndarray    # [B,n_eval,5,N]
    t: np.ndarray            # [B] time reached
    status: np.ndarray       # [B]
    n_accepted: np.ndarray
    n_rejected: np.ndarray
    nfev: np.ndarray
    event_counts: np.ndarray  # [B,7]
    owner: np.ndarray        # [B] rank that integrated the column
    t_eval: np.ndarray
    next_eval: np.ndarray = None   # [B] rows of `snapshots` that hold data (the rest is NaN: column stopped early)


def sweep_radau(pde: dict, **kw) -> SweepResult:
    """The sweep with the implicit integrator (the reference's default Solver, parameters.py:207-221): what a
    65 536-column sweep to T* uses in practice (4096 columns: ~23 s against ~140 s with RK45)."""
    return sweep_rk45(pde, method="Radau", **kw)


def sweep_bdf(pde: dict, **kw) -> SweepResult:
    """The sweep with the variable-order BDF kernel (solve_ivp(method="BDF"), parameters.py:235-236; LSODA's stiff mode)."""
    return sweep_rk45(pde, method="BDF", **kw)


def sweep_rk45(pde: dict, t_span=(0.0, 1.0), first_step=1e-6, rtol=1e-3, atol=1e-3, t_eval=None,
               events: bool = True, balance: bool = True, group=None, device=None, integrate=None,
               method: str = "RK45", **kw) -> SweepResult:
    """Integrate every column of the sweep dictionary `pde` with the on-device RK45 (or the integrator `method` names:
    "RK23", "DOP853", "Radau", "BDF"), sharded over the ranks of `group` (all ranks call this with the same arguments).  `integrate` is the
    per-rank batched integrator (default: marlpde_b200.integrate_{rk45,radau}_batch on `device`)."""
    import torch
    import torch.distributed as dist
    from . import params as _params

    ddp = dist.is_available() and dist.is_initialized()
    world = dist.get_world_size(group) if ddp else 1
    rank = dist.get_rank(group) if ddp else 0
    B = n_columns_of(pde)
    if balance and world > 1:
        assign = balanced_assignment(predicted_cost(pde, method) * np.ones(B), world)
    else:
        assign = [np.arange(a, b, dtype=np.int64) for a, b in partition(B, world)]
    mine = assign[rank]
    counts = [len(a) for a in assign]
    local = shard(pde, mine) if B > 1 else pde

    if integrate is None:
        from .batch import (integrate_bdf_batch, integrate_dop853_batch, integrate_radau_batch, integrate_rk23_batch,
                            integrate_rk45_batch)
        run = {"RK45": integrate_rk45_batch, "RK23": integrate_rk23_batch, "DOP853": integrate_dop853_batch,
               "Radau": integrate_radau_batch, "BDF": integrate_bdf_batch}.get(method)
        if run is None:
            raise ValueError("method must be 'RK45', 'RK23', 'DOP853', 'Radau' or 'BDF'")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)

        def integrate(y0, P, **opts):
            return run(torch.from_numpy(y0).to(dev), P, **opts)
    P = _params.derive_column_params(local) if len(mine) else None
    te = np.zeros(0) if t_eval is None else np.asarray(t_eval, dtype=np.float64)
    N = int(pde["N"])
    if len(mine):
        res = integrate(_params.initial_state(local), P, t_span=t_span, first_step=first_step, rtol=rtol,
                        atol=atol, t_eval=t_eval, events=events, **kw)
        as_t = lambda a: a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a))  # noqa: E731
        y_l, snap_l = as_t(res.y), as_t(res.snapshots)
        stats = np.stack([res.t, res.status.astype(np.float64), res.n_accepted.astype(np.float64),
                          res.n_rejected.astype(np.float64), res.nfev.astype(np.float64)], axis=1)
        stats = np.concatenate([stats, np.asarray(res.event_counts, dtype=np.float64).reshape(len(mine), 7),
                                np.asarray(getattr(res, "next_eval", np.full(len(mine), te.size)), dtype=np.float64)[:, None]],
                               axis=1)
        dev_l = y_l.device
    else:
        dev_l = torch.device("cuda", torch.cuda.current_device()) if (device is None and torch.cuda.is_available()) \
            else torch.device(device or "cpu")
        y_l = torch.zeros((0, 5, N), dtype=torch.float64, device=dev_l)
        snap_l = torch.zeros((0, te.size, 5, N), dtype=torch.float64, device=dev_l)
        stats = np.zeros((0, 13))
    stats_l = torch.from_numpy(stats).to(dev_l)

    # ---- the one collective: end states, snapshots and per-column statistics of every shard
    y_all = gather_columns(y_l, counts, group)
    snap_all = gather_columns(snap_l, counts, group)
    stats_all = gather_columns(stats_l, counts, group)
    order = np.concatenate(assign) if world > 1 else mine           # gathered row -> original column
    inv = np.empty(B, dtype=np.int64)
    inv[order] = np.arange(B)
    y_np = y_all.cpu().numpy()[inv]
    snap_np = snap_all.cpu().numpy()[inv]
    st = stats_all.cpu().numpy()[inv]
    owner = np.empty(B, dtype=np.int64)
    for r, a in enumerate(assign):
        owner[a] = r
    return SweepResult(y=y_np, snapshots=snap_np, t=st[:, 0], status=st[:, 1].astype(np.int32),
                       n_accepted=st[:, 2].astype(np.int64), n_rejected=st[:, 3].astype(np.int64),
                       nfev=st[:, 4].astype(np.int64), event_counts=st[:, 5:12].astype(np.int64), owner=owner,
                       t_eval=te, next_eval=st[:, 12].astype(np.int64))
