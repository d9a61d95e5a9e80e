"""Host side of the BDF integrator's forward sensitivities: the parameter directions of
marlpde_b200.sensitivity_directions (no GPU needed)."""
import numpy as np
import pytest

import lheureux_oracle as oracle
import marlpde_b200 as mb


def test_k2_moves_exactly_Da_lambda_and_nu1():
    """k2 enters Da = k2 Tstar, lambda = k3 / k2 and nu1 = k1 / k2 and nothing else; (Da+ - Da-) inv2sigma = Tstar."""
    pde = oracle.default_scenario()
    sd = mb.sensitivity_directions(pde, ["k2"])
    p = mb.derive_column_params(pde)[0]
    pp, pn = sd.params_pm[0, 0, 0], sd.params_pm[0, 0, 1]
    moved = {f for f in p.dtype.names if not (np.array_equal(pp[f], p[f]) and np.array_equal(pn[f], p[f]))}
    assert moved == {"Da", "lambda_", "nu1"}
    assert abs((pp["Da"] - pn["Da"]) * sd.inv2sigma[0, 0] / pde["Tstar"] - 1.0) <= 1e-9
    assert np.all(sd.w == 0.0)


def test_PhiIni_direction_moves_the_initial_porosity():
    """PhiIni gives w = 1 on the Phi rows and 0 elsewhere (and moves dPhi_fixed, which depends on PhiIni)."""
    pde = oracle.default_scenario()
    sd = mb.sensitivity_directions(pde, ["PhiIni"])
    w = sd.w[0, 0]
    assert np.all(w[:4] == 0.0)
    assert np.max(np.abs(w[4] - 1.0)) <= 1e-9
    assert sd.params_pm[0, 0, 0]["dPhi_fixed"] != sd.params_pm[0, 0, 1]["dPhi_fixed"]


def test_linear_combination_over_a_sweep():
    """A {key: coefficient} direction with per-column coefficients: the consistent S direction of a lattice sweep moves
    Tstar by -2 D0Ca / S^3 per unit, so Da moves by k2 times that."""
    lat = mb.sweep_lattice(oracle.default_scenario(), 2, 1, 2)
    S, D0Ca = lat["sedimentationrate"], lat["D0Ca"]
    sd = mb.sensitivity_directions(lat, [{"sedimentationrate": 1.0, "Xstar": -D0Ca / S ** 2, "Tstar": -2 * D0Ca / S ** 3}])
    assert sd.params_pm.shape == (4, 1, 2) and sd.names == ["sedimentationrate+Xstar+Tstar"]
    dDa = (sd.params_pm[:, 0, 0]["Da"] - sd.params_pm[:, 0, 1]["Da"]) * sd.inv2sigma[:, 0]
    assert np.allclose(dDa, lat["k2"] * (-2 * D0Ca / S ** 3), rtol=1e-8)
    assert np.allclose(sd.atol(1e-3), 1e-3 / sd.pbar) and np.all(sd.pbar > 0)


def test_mask_boundary_on_the_switching_point_is_refused():
    """A ShallowLimit that sits where the dissolution mask switches (on a cell centre: cell i is inside when its centre
    is strictly below the limit) moves a mask boundary within +/- sigma: ValueError naming the direction."""
    pde = oracle.default_scenario()
    dx = pde["max_depth"] / pde["N"]
    at_centre = pde | {"ShallowLimit": 20.5 * dx}
    with pytest.raises(ValueError, match="ShallowLimit"):
        mb.sensitivity_directions(at_centre, ["ShallowLimit"])
    mb.sensitivity_directions(pde | {"ShallowLimit": 20.0 * dx + 0.3 * dx}, ["ShallowLimit"])   # away from it: fine


@pytest.mark.parametrize("wrt", [["N"], ["FV_switch"], [{"k2": 1.0, "N": 1.0}], ["k1"] * 9, []])
def test_refused_directions(wrt):
    """N and FV_switch are not continuous parameters; 1 to 8 directions."""
    with pytest.raises(ValueError):
        mb.sensitivity_directions(oracle.default_scenario(), wrt)


def test_sensitivity_entry_points_are_exported():
    """The C ABI carries the sensitivity entry points next to the BDF ones."""
    from marlpde_b200 import _cabi
    lib = _cabi.lib()
    assert lib.marlpde_bdf_sens_workspace_bytes(4, 200, 3) == 8 * 4 * (140 * 200 + 3 * 60 * 200)
    assert lib.marlpde_bdf_sens_workspace_bytes(4, 200, 0) == 0
