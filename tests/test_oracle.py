"""The CPU oracle against the golden vectors produced by the unmodified reference (oracle/make_golden.py)."""
import numpy as np
import pytest

import gp_oracle as orc
from conftest import REAL_CONFIGS, load_golden

COND_OK = 1e8


def rel(a, b, scale=None):
    a, b = np.asarray(a), np.asarray(b)
    s = np.abs(b).max() if scale is None else scale
    return np.abs(a - b).max() / max(s, 1e-300)


def test_fixed_theta_numpy_restatement():
    g = load_golden("fixed_theta_synth")
    for m in g["sizes"]:
        t, y = g[f"t_{m}"], g[f"y_{m}"]
        for gi in range(2):
            for k, th in enumerate(g["thetas"]):
                if g[f"cond_{m}"][gi, k] > COND_OK:
                    continue
                lml, grad, st = orc.np_lml_grad(t, y[gi], th)
                assert st == 0
                assert abs(lml - g[f"lml_{m}"][gi, k]) <= 1e-10 * abs(g[f"lml_{m}"][gi, k])
                ref = g[f"grad_{m}"][gi, k]
                assert rel(grad, ref) <= 1e-9


def test_synthetic_generator_is_the_goldens_input():
    g = load_golden("fixed_theta_synth")
    t, y = orc.synthetic_trajectories(2, 200, seed=200)
    assert np.array_equal(t, g["t_200"]) and np.array_equal(y, g["y_200"])


@pytest.mark.parametrize("name", REAL_CONFIGS)
def test_real_config_fixed_theta(name):
    g = load_golden(name)
    T, Y = g["T"], g["Y"]
    for gi in range(T.shape[0]):
        for k, th in enumerate(g["thetas_eval"][gi]):
            if g["cond_eval"][gi, k] > COND_OK or not np.isfinite(g["lml_eval"][gi, k]):
                continue
            lml, grad, st = orc.np_lml_grad(T[gi], Y[gi], th)
            assert abs(lml - g["lml_eval"][gi, k]) <= 1e-10 * max(1.0, abs(g["lml_eval"][gi, k]))
            assert rel(grad, g["grad_eval"][gi, k], max(1.0, np.abs(g["grad_eval"][gi, k]).max())) <= 1e-8


@pytest.mark.parametrize("name", REAL_CONFIGS)
def test_real_config_moments(name):
    g = load_golden(name)
    T, Y, t_est, eta = g["T"], g["Y"], g["t_est"], float(g["eta"])
    for gi in range(min(T.shape[0], 3)):
        th = g["theta_opt"][gi]
        alpha, _ = orc.np_alpha(T[gi], Y[gi], th)
        assert rel(alpha, g["alpha_opt"][gi]) <= 1e-9
        mean, std = orc.np_predict(T[gi], Y[gi], th, t_est)
        assert rel(mean, g["pred_mean"][gi]) <= 1e-10
        assert rel(std, g["pred_std"][gi]) <= 1e-8
        out = orc.np_lstsq_moments(T[gi], Y[gi], th, t_est, eta, want_sqrtW=False)
        assert rel(out["state_estimate"], g["state_estimate"][gi]) <= 1e-10
        assert rel(out["ddt_estimate"], g["ddt_estimate"][gi]) <= 1e-10
        if gi < g["ddt_covariance"].shape[0]:
            assert rel(out["ddt_covariance"], g["ddt_covariance"][gi]) <= 1e-9


def test_oracle_gp_port_reproduces_reference_fit():
    """OracleGP (sklearn-driven port of GP_RBFW) with the reference's RNG contract reproduces the golden optimum."""
    g = load_golden("heat_1_20_05_80_5")
    b = g["bounds"]
    gi = 0
    # replay the restart points through the global RNG: OracleGP draws them exactly like the reference
    class _Replay:
        def __init__(self, pts):
            self.pts, self.k = pts, 0

        def uniform(self, lo, hi):
            p = self.pts[self.k]
            self.k += 1
            return p

    gp = orc.OracleGP(tuple(b[0]), tuple(b[1]), tuple(b[2]), int(g["n_restarts"]))
    gp.gpr.random_state = None
    import sklearn.utils

    orig = sklearn.gaussian_process._gpr.check_random_state
    sklearn.gaussian_process._gpr.check_random_state = lambda rs: _Replay(g["starts"][gi])
    try:
        gp.fit(g["T"][gi], g["Y"][gi])
    finally:
        sklearn.gaussian_process._gpr.check_random_state = orig
    assert abs(gp.lml - g["lml_opt"][gi]) <= 1e-9 * abs(g["lml_opt"][gi])
    assert np.allclose(gp.theta, g["theta_opt"][gi], atol=1e-4)


def test_reference_import_matches_oracle():
    """The oracle against what the unmodified reference's GP_RBFW returned when the goldens were made
    (oracle/make_golden.py): ``gp.gpr.log_marginal_likelihood(theta, eval_gradient=True)`` on synthetic data at
    m = 64, and ``compute_lstsq_matrices(t_est, eta=1e-8)`` at the fitted theta of the Heat configuration."""
    g = load_golden("fixed_theta_synth")
    t, y = g["t_64"], g["y_64"]
    checked = 0
    for gi in range(2):
        for k, th in enumerate(g["thetas"]):
            if g["cond_64"][gi, k] > COND_OK:
                continue
            l_ref, g_ref = g["lml_64"][gi, k], g["grad_64"][gi, k]
            l, gr, _ = orc.np_lml_grad(t, y[gi], th)
            assert abs(l - l_ref) <= 1e-11 * abs(l_ref)
            assert rel(gr, g_ref) <= 1e-9
            checked += 1
    assert checked >= 4
    h = load_golden("heat_1_20_05_80_5")
    assert float(h["eta"]) == 1e-8
    for gi in range(h["ddt_covariance"].shape[0]):
        out = orc.np_lstsq_moments(h["T"][gi], h["Y"][gi], h["theta_opt"][gi], h["t_est"], 1e-8, want_sqrtW=False)
        assert rel(out["ddt_covariance"], h["ddt_covariance"][gi]) <= 1e-10
        assert rel(out["ddt_estimate"], h["ddt_estimate"][gi]) <= 1e-11


# ------------------------------------------------------------------ Matern extension of the oracle
@pytest.mark.parametrize("twice_nu", [3, 5])
def test_matern_oracle_formulas(twice_nu):
    """np_matern against scikit-learn's Matern, its derivatives against central differences."""
    rng = np.random.default_rng(twice_nu)
    t1, t2 = np.sort(rng.uniform(0, 1, 40)), np.sort(rng.uniform(0, 1, 31))
    th = np.log([1.3, 0.2, 1e-3])
    sk = orc.sk_matern_kernel(th, twice_nu)
    assert rel(orc.np_matern(t1, t2, 1.3, 0.2, twice_nu), sk(t1[:, None], t2[:, None])) <= 1e-14
    h = 1e-5
    k = lambda a, b: orc.np_matern(a, b, 1.3, 0.2, twice_nu)
    d1 = (k(t1 + h, t2) - k(t1 - h, t2)) / (2 * h)
    far = np.abs(t1[:, None] - t2[None, :]) > 10 * h
    assert np.abs(d1 - orc.np_matern(t1, t2, 1.3, 0.2, twice_nu, deriv=1))[far].max() <= 1e-7 * np.abs(d1).max()
    d2 = (k(t1 + h, t2 + h) - k(t1 + h, t2 - h) - k(t1 - h, t2 + h) + k(t1 - h, t2 - h)) / (4 * h * h)
    assert np.abs(d2 - orc.np_matern(t1, t2, 1.3, 0.2, twice_nu, deriv=2))[far].max() <= 1e-4 * np.abs(d2).max()
    # LML / gradient restatement against sklearn's own regressor
    y = np.sin(7 * t1) + 0.05 * rng.standard_normal(40)
    gp = orc.OracleGP((1e-5, 1e5), (1e-5, 1e2), (1e-16, 1e2), 0, twice_nu=twice_nu)
    gp.gpr.optimizer = None
    gp.fit(t1, y)
    l_ref, g_ref = gp.lml_grad(th)
    l, g, st = orc.np_lml_grad_matern(t1, y, th, twice_nu)
    assert st == 0 and abs(l - l_ref) <= 1e-12 * abs(l_ref) and rel(g, g_ref) <= 1e-10


def test_lean_restatement_equals_full_restatement():
    """np_lml_grad_lean (used for the m = 16384 golden) against np_lml_grad and the reference goldens."""
    g = load_golden("fixed_theta_synth")
    m = 512
    t, y = g[f"t_{m}"], g[f"y_{m}"]
    for k, th in enumerate(g["thetas"][:4]):
        a = orc.np_lml_grad(t, y[0], th)
        b = orc.np_lml_grad_lean(t, y[0], th, block=200, want_alpha=True)
        assert a[2] == b[2] == 0
        assert abs(a[0] - b[0]) <= 1e-13 * abs(a[0])
        assert rel(b[1], a[1]) <= 1e-12
        assert abs(b[0] - g[f"lml_{m}"][0, k]) <= 1e-10 * abs(g[f"lml_{m}"][0, k])
    # all-equal abscissae, chi below one ulp of sigma^2: exact zero pivot -> status 1 like np_lml_grad
    assert orc.np_lml_grad_lean(np.full(64, 0.5), np.linspace(-1, 1, 64), np.log([1.0, 0.1, 1e-17]))[2] == 1


def test_large_golden_is_self_consistent():
    """fixed_theta_large.npz: the lean restatement agreed with the unmodified reference at m = 4096 when the file was
    made, and the reference is within cond * eps of the 80-bit truth."""
    import os

    from conftest import GOLDEN

    if not os.path.isfile(os.path.join(GOLDEN, "fixed_theta_large.npz")):
        pytest.skip("not generated")
    g = load_golden("fixed_theta_large")
    assert np.all(g["lean_vs_reference_rel"] <= 1e-11)
    for m in g["sizes"]:
        if f"truth_lml_{m}" not in g.files:
            continue
        tl, rl = g[f"truth_lml_{m}"], g[f"lml_{m}"]
        done = tl != 0.0
        assert np.all(np.abs(tl[done] - rl[done]) <= 1e-11 * np.abs(tl[done]))
        cond = g[f"cond_{m}"][done]
        ea = np.abs(g[f"truth_alpha_{m}"][done] - g[f"alpha_{m}"][done]).max(1) / np.abs(g[f"truth_alpha_{m}"][done]).max(1)
        assert np.all(ea <= 1e-15 * cond * 10)


def test_long_double_truth_matches_numpy():
    """oracle/lml_ld.c (80-bit) against the FP64 restatement at a size where FP64 is accurate to ~1e-13."""
    import os
    import shutil
    import subprocess

    from conftest import ROOT

    if shutil.which("gcc") is None:
        pytest.skip("needs gcc")
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle")], check=True, capture_output=True)
    t, y = orc.synthetic_trajectories(1, 256, seed=3)
    th = np.log([1.3, 0.08, 2e-3])
    l, g, a = orc.ld_truth(t, y[0], th)
    l0, g0, _ = orc.np_lml_grad(t, y[0], th)
    a0, _ = orc.np_alpha(t, y[0], th)
    assert abs(l - l0) <= 1e-12 * abs(l0) and rel(g, g0) <= 1e-11 and rel(a, a0) <= 1e-10
    l, g, a = orc.ld_truth(np.full(16, 0.5), np.linspace(-1, 1, 16), np.log([1.0, 0.1, 1e-25]))
    assert l == -np.inf and np.all(g == 0)


def test_package_workload_equals_the_goldens_generator():
    from gpbo_pkg import pkg

    t, y = orc.synthetic_trajectories(3, 77, seed=5)
    t2, y2 = pkg.workload.synthetic_trajectories(3, 77, seed=5)
    assert np.array_equal(t, t2) and np.array_equal(y, y2)
    T, Y, bl, starts, gp_of = pkg.workload.fit_workload(3, 77, 4, seed=5)
    assert T.shape == Y.shape == (3, 77) and starts.shape == (12, 3) and np.all(starts[::4] == 0)
    assert np.all((starts >= bl[:, 0]) & (starts <= bl[:, 1])) and gp_of.tolist() == [0] * 4 + [1] * 4 + [2] * 4
