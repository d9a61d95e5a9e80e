"""marlpde_b200 — host side of the B200-native integrator for L'Heureux's diagenetic model.

Layers (bottom up):
  csrc/ + include/marlpde_b200.h   hand-written sm_100a kernels behind a C ABI
  _cabi                            ctypes binding of that ABI
  params                           per-column constants (mirror of LMAHeureuxPorosityDiff.__init__)
  sensitivity                      parameter directions of the BDF integrator's forward sensitivities
  batch                            batched RHS / RK45 entry points on host or device buffers
  sweep                            column sharding over GPUs + the one all-gather of results
  pde_standin, hdf5lite            the sliver of py-pde / h5py the reference driver touches
The reference-facing drop-in (`Map_Scenario`, `Solver`, `Tracker`, `LMAHeureuxPorosityDiff`,
`integrate_equations`) lives in the sibling package `marlpde`.
"""
from . import _cabi  # noqa: F401
from .params import derive_column_params, initial_state, sweep_lattice  # noqa: F401
from .batch import rhs_batch, integrate_rk45_batch, integrate_radau_batch, integrate_bdf_batch, RK45Result, RadauResult  # noqa: F401
from .batch import integrate_rk23_batch, integrate_dop853_batch  # noqa: F401
from .sensitivity import sensitivity_directions, SensitivityDirections  # noqa: F401
from . import sweep  # noqa: F401
