"""The library's L-BFGS-B state machine (host-only entry point) against scipy's L-BFGS-B."""
import numpy as np
import pytest
import scipy.optimize as so

import gp_oracle as orc
from conftest import load_golden
from gpbo_pkg import pkg

BOX = np.array([[-3.0, 3.0], [-2.0, 4.0], [-5.0, 1.0]])


def quad(x):
    A = np.array([[3.0, 0.5, 0.1], [0.5, 2.0, -0.3], [0.1, -0.3, 1.0]])
    b = np.array([1.0, -2.0, 0.5])
    return 0.5 * x @ A @ x - b @ x, A @ x - b


def rosen3(x):
    f = so.rosen(x)
    return f, so.rosen_der(x)


def active_bound(x):
    c = np.array([5.0, -4.0, 0.3])       # unconstrained minimiser outside the box in two coordinates
    return float(((x - c) ** 2).sum()), 2 * (x - c)


@pytest.mark.parametrize("fn", [quad, rosen3, active_bound])
def test_matches_scipy_on_analytic_functions(fn):
    rng = np.random.default_rng(0)
    for _ in range(10):
        x0 = rng.uniform(BOX[:, 0], BOX[:, 1])
        mine = pkg._lib.lbfgsb_minimize(fn, x0, BOX)
        ref = so.minimize(fn, x0, method="L-BFGS-B", jac=True, bounds=BOX)
        assert mine["status"] in (0, 1)
        assert mine["fun"] <= ref.fun + 1e-8 * max(1.0, abs(ref.fun))
        assert np.allclose(mine["x"], ref.x, atol=2e-4)
        assert mine["nfev"] <= 2 * ref.nfev + 5


def test_start_outside_box_is_clipped_like_scipy():
    x0 = np.array([10.0, -10.0, 0.0])
    mine = pkg._lib.lbfgsb_minimize(quad, x0, BOX)
    ref = so.minimize(quad, x0, method="L-BFGS-B", jac=True, bounds=BOX)
    assert np.allclose(mine["x"], ref.x, atol=1e-5)


def test_empty_bound_interval_is_rejected():
    """lo > hi in any coordinate is an argument error, as in gpbo_optpool_create and gpbo_fit_host."""
    for i in range(3):
        box = BOX.copy()
        box[i] = box[i, ::-1]
        with pytest.raises(pkg.GpboError, match="status -1.*empty bound interval"):
            pkg._lib.lbfgsb_minimize(quad, np.zeros(3), box)


def test_non_finite_start_terminates():
    r = pkg._lib.lbfgsb_minimize(lambda x: (np.inf, np.zeros(3)), np.zeros(3), BOX)
    assert r["status"] == 5 and r["nfev"] == 1


def test_best_of_starts_reaches_reference_optimum_on_heat():
    """Optimiser parity gate (BASELINE.json: optimum LML within 1e-8 relative of the reference's), on the
    CPU with the oracle as objective and the reference's own restart points."""
    g = load_golden("heat_1_20_05_80_5")
    bl = np.log(g["bounds"])
    for gi in (0, 7):
        t, y = g["T"][gi], g["Y"][gi]

        def f(x):
            l, gr, _ = orc.np_lml_grad(t, y, x)
            return -l, -gr

        S = np.vstack([np.zeros((1, 3)), g["starts"][gi]])
        best = min(pkg._lib.lbfgsb_minimize(f, s, bl)["fun"] for s in S)
        assert abs(-best - g["lml_opt"][gi]) <= 1e-8 * abs(g["lml_opt"][gi])
