"""Parameter directions for the forward sensitivities of the BDF integrator (csrc/bdf_batch.cu, DESIGN.md 5.4).

A direction is a perturbation of the reference's `pde_parms` dictionary: one key, or a linear combination
{key: coefficient, ...}.  Moving along it by eps moves the derived column parameters p (and the initial state y0); the
kernel integrates s = dy/d eps with F = df/d eps formed as a central difference of the RHS between the parameter sets
p(+sigma) and p(-sigma) that this module derives on the host — the kernel never differentiates a parameter record.

Derivatives are taken at fixed NONDIMENSIONAL time t (= t_years / Tstar, the time the kernels integrate in): a direction
that moves Tstar (through `sedimentationrate`, `D0Ca`, or `Tstar` itself) gives dy(t)/d eps at fixed t, not at fixed
years.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Mapping, Sequence

import numpy as np

from .params import _n_columns, derive_column_params, initial_state

MAX_DIRECTIONS = 8
_INT_FIELDS = ("FV_switch", "mask_lo", "mask_hi", "model_flags")
_FORBIDDEN = ("N", "FV_switch")


@dataclass
class SensitivityDirections:
    """Host-derived inputs of the sensitivity kernel for B columns and P directions."""
    names: list                  # [P] direction names
    params_pm: np.ndarray        # (B, P, 2) marlpde_column_params: p moved by +sigma and by -sigma
    inv2sigma: np.ndarray        # (B, P) 1 / (2 sigma)
    w: np.ndarray                # (B, P, 5, N) dy0 / d eps (central difference of initial_state)
    pbar: np.ndarray             # (B, P) size of the direction's entries (sigma = eps^(1/3) pbar)

    @property
    def n_dirs(self) -> int:
        return len(self.names)

    def atol(self, atol: float) -> np.ndarray:
        """Default absolute tolerance of s in the corrector: atol / pbar per column and direction (CVODES' pbar
        scaling: s pbar is measured in the units of y)."""
        return np.ascontiguousarray(float(atol) / self.pbar)


def _as_direction(item) -> tuple[str, dict]:
    if isinstance(item, str):
        return item, {item: 1.0}
    if isinstance(item, Mapping):
        if not item:
            raise ValueError("an empty direction")
        return "+".join(str(k) for k in item), dict(item)
    raise TypeError(f"a direction is a key of pde or a {{key: coefficient}} dict, not {item!r}")


def sensitivity_directions(pde: Mapping, wrt: Sequence, eps: float | None = None) -> SensitivityDirections:
    """Derive the kernel inputs for the directions `wrt` (at most 8): each item is a key of `pde` or a dict
    {key: coefficient} (a coefficient may be an array over the sweep's columns).  Example — the sedimentation rate S
    moved consistently with what Map_Scenario derives from it (Xstar = D0Ca / S, Tstar = Xstar / S):
    {"sedimentationrate": 1, "Xstar": -D0Ca / S**2, "Tstar": -2 * D0Ca / S**3}.

    sigma = eps^(1/3) pbar with pbar = min over the entries of |pde[key]| / |coefficient| (entries whose value is 0 are
    skipped; pbar = 1 if all are); p+/- = derive_column_params(pde +/- sigma dir), w = the central difference of
    initial_state.  Raises ValueError, naming the direction, for the keys N and FV_switch and when p+ or p- differs from
    p in an integer field (a mask boundary moved: the state is not differentiable there)."""
    wrt = list(wrt)
    if not 1 <= len(wrt) <= MAX_DIRECTIONS:
        raise ValueError(f"between 1 and {MAX_DIRECTIONS} sensitivity directions are supported (got {len(wrt)})")
    eps = np.finfo(np.float64).eps if eps is None else float(eps)
    B = _n_columns(pde)
    N = int(pde["N"])
    p0 = derive_column_params(pde)
    names, pm, inv2s, ws, pbars = [], [], [], [], []
    for item in wrt:
        name, coef = _as_direction(item)
        for key in coef:
            if key in _FORBIDDEN:
                raise ValueError(f"direction {name!r}: {key!r} is not a continuous parameter")
            if key not in pde:
                raise ValueError(f"direction {name!r}: {key!r} is not a parameter of the scenario")
        pbar = np.full(B, np.inf)
        for key, c in coef.items():
            v = np.abs(np.broadcast_to(np.asarray(pde[key], dtype=np.float64), (B,)))
            c = np.abs(np.broadcast_to(np.asarray(c, dtype=np.float64), (B,)))
            with np.errstate(divide="ignore", invalid="ignore"):
                r = np.where((v > 0) & (c > 0), v / c, np.inf)
            pbar = np.minimum(pbar, r)
        pbar = np.where(np.isfinite(pbar), pbar, 1.0)
        sigma = np.cbrt(eps) * pbar
        moved = []
        for sign in (1.0, -1.0):
            q = dict(pde)
            for key, c in coef.items():
                q[key] = np.asarray(pde[key], dtype=np.float64) + sign * sigma * np.asarray(c, dtype=np.float64)
            moved.append(q)
        pp, pn = derive_column_params(moved[0]), derive_column_params(moved[1])
        for f in _INT_FIELDS:
            if np.any(pp[f] != p0[f]) or np.any(pn[f] != p0[f]):
                raise ValueError(f"direction {name!r} changes the integer field {f} of some columns (a mask boundary or "
                                 "switch moves within +/- sigma): the state is not differentiable in this direction there")
        i2s = 1.0 / (2.0 * sigma)
        w = (initial_state(moved[0]) - initial_state(moved[1])) * i2s[:, None, None]
        names.append(name)
        pm.append(np.stack([pp, pn], axis=1))
        inv2s.append(i2s)
        ws.append(w)
        pbars.append(pbar)
    return SensitivityDirections(names=names, params_pm=np.ascontiguousarray(np.stack(pm, axis=1)),
                                 inv2sigma=np.ascontiguousarray(np.stack(inv2s, axis=1)),
                                 w=np.ascontiguousarray(np.stack(ws, axis=1).reshape(B, len(wrt), 5, N)),
                                 pbar=np.ascontiguousarray(np.stack(pbars, axis=1)))
