"""Every run-time switch of DESIGN.md §11 is still read and still does what the table says.  The library reads the
switches once per process, so each run is a child process (this file run as a script) with one switch set; it prints
its results and the per-class launch counts, and its stderr is kept."""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M = 1000                                    # blocked path, T = 8 block columns
T_BLOCKS = 8


def _workload(name):
    """Run one workload on a fresh context; returns (arrays, per-class launch counts)."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gp_oracle as orc
    from gpbo_pkg import pkg

    ctx = pkg.Context(0)
    ctx.profile_enable(True)
    if name in ("lml", "lml1", "small"):
        B = {"lml": 4, "lml1": 1, "small": 4}[name]
        m = 90 if name == "small" else M
        t, y = orc.synthetic_trajectories(B, m, seed=11)
        theta = np.random.default_rng(11).uniform(np.log([0.3, 0.01, 1e-2]), np.log([3.0, 0.1, 1e-1]), size=(B, 3))
        lml, grad, st = ctx.lml_grad(np.tile(t, (B, 1)), y, theta)
        out = dict(lml=lml, grad=grad, status=st)
    elif name in ("predict", "lstsq"):
        G = 4 if name == "predict" else 2
        t, y = orc.synthetic_trajectories(G, M, seed=12)
        theta = np.tile(np.log([1.5, 0.05, 1e-2]), (G, 1))
        if name == "predict":                                 # 4 GPs x 64 row tiles: enough for the row sweep
            mean, std, _, st = ctx.predict(np.tile(t, (G, 1)), y, theta, np.linspace(0.0, 1.0, 8192))
            out = dict(mean=mean, std=std, status=st)
        else:                                                 # equispaced: the Toeplitz K_zz table applies
            state, ddt, cov, st = ctx.lstsq_moments(np.tile(t, (G, 1)), y, theta, np.linspace(0.0, 1.0, 300))
            out = dict(state=state, ddt=ddt, cov=cov, status=st)
    elif name == "sqrtw":                                     # condition number 1e3, eta = 1e-3
        n = 64
        q, _ = np.linalg.qr(np.random.default_rng(13).standard_normal((n, n)))
        cov = (q * np.logspace(-3.0, 0.0, n)) @ q.T
        w, st, it = ctx.sqrtw(0.5 * (cov + cov.T), 1e-3)
        out = dict(sqrtw=w, status=st, iters=it)
    else:
        raise ValueError(name)
    counts = {k: n for k, (_, n) in ctx.profile_get().items()}
    ctx.close()
    return {k: np.asarray(v).tolist() for k, v in out.items()}, counts


@functools.lru_cache(maxsize=None)
def run(name, **env):
    e = dict(os.environ)
    for k in list(e):
        if k.startswith("GPBO_") and k != "GPBO_LIB":
            del e[k]
    e.update(env)
    p = subprocess.run([sys.executable, os.path.abspath(__file__), name], env=e, capture_output=True, text=True,
                       timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    out, counts = json.loads(p.stdout.strip().splitlines()[-1])
    return {k: np.array(v) for k, v in out.items()}, counts, p.stderr


def rel(a, b):
    return float(np.abs(a - b).max() / max(1e-300, np.abs(b).max()))


@pytest.mark.gpu
def test_no_sweep_runs_per_column_launches():
    (d, dc, _), (s, sc, _) = run("predict"), run("predict", GPBO_NO_SWEEP="1")
    assert dc["cross_panel"] == 1 and sc["cross_panel"] >= T_BLOCKS, (dc, sc)
    assert rel(s["mean"], d["mean"]) <= 1e-10 and rel(s["std"], d["std"]) <= 1e-8


@pytest.mark.gpu
def test_sweep_mode_stays_within_tolerance():
    (d, dc, _), (s, sc, _) = run("predict"), run("predict", GPBO_SWEEP_MODE="1")
    assert sc == dc
    assert rel(s["mean"], d["mean"]) <= 1e-10 and rel(s["std"], d["std"]) <= 1e-8


@pytest.mark.gpu
def test_no_toeplitz_drops_the_kzz_table():
    (d, dc, _), (s, sc, _) = run("lstsq"), run("lstsq", GPBO_NO_TOEPLITZ="1")
    assert dc["prep"] - sc["prep"] == 1, (dc, sc)            # one wave: one kzz_table launch fewer
    assert rel(s["state"], d["state"]) <= 1e-10 and rel(s["ddt"], d["ddt"]) <= 1e-10
    assert rel(s["cov"], d["cov"]) <= 1e-9


@pytest.mark.gpu
def test_split_max_one_removes_split_k_partials():
    (d, dc, _) = run("lml1")
    (s, sc, _) = run("lml1", GPBO_SPLIT_MAX="1", GPBO_NO_QUANT_SPLIT="1")
    # one launch per block column left: T - 1 panels, T - 1 inverse rows
    assert sc["chol_panel"] == T_BLOCKS - 1 and sc["trtri"] == T_BLOCKS - 1, sc
    assert dc["chol_panel"] > sc["chol_panel"] and dc["trtri"] > sc["trtri"], dc
    _within_lml_tolerance(s, d)


def _within_lml_tolerance(s, d):
    assert np.array_equal(s["status"], d["status"]) and not d["status"].any()
    assert np.all(np.abs(s["lml"] - d["lml"]) <= 1e-10 * np.abs(d["lml"]))
    for g, g0 in zip(s["grad"], d["grad"]):
        assert np.abs(g - g0).max() <= 1e-9 * max(1.0, np.abs(g0).max())


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"GPBO_OVERLAP_MAX": "0"}, {"GPBO_SIDE_SPLIT_DIV": "1"}, {"GPBO_TRTRI_LPT": "0"}])
def test_schedule_switches_are_bit_identical(env):
    (d, dc, _), (s, sc, _) = run("lml"), run("lml", **env)
    assert sc == dc
    for k in ("lml", "grad", "status"):
        assert np.array_equal(s[k], d[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"GPBO_NO_TMA": "1"}, {"GPBO_SIDE_SPLIT_DIV": "4"}, {"GPBO_SPLIT_MIN": "8"},
                                 {"GPBO_SPLIT_MAX": "4"}, {"GPBO_NO_QUANT_SPLIT": "1"}])
def test_tuning_switches_stay_within_tolerance(env):
    _within_lml_tolerance(run("lml", **env)[0], run("lml")[0])


@pytest.mark.gpu
def test_ns_plain_needs_more_iterations():
    (d, _, _), (s, _, _) = run("sqrtw"), run("sqrtw", GPBO_NS_PLAIN="1")
    assert not d["status"].any() and not s["status"].any()
    assert s["iters"][0] > d["iters"][0], (s["iters"], d["iters"])
    assert rel(s["sqrtw"], d["sqrtw"]) <= 1e-8


@pytest.mark.gpu
def test_debug_switches_print_to_stderr():
    assert "[gpbo sqrtw] it 0 " not in run("sqrtw")[2]
    assert "[gpbo sqrtw] it 0 " in run("sqrtw", GPBO_DEBUG_NS="1")[2]
    assert "[gpbo small lml_grad m=90] cycles:" not in run("small")[2]
    (s, _, err) = run("small", GPBO_SMALL_DBG="1")
    assert "[gpbo small lml_grad m=90] cycles:" in err
    assert not s["status"].any()


if __name__ == "__main__":
    print(json.dumps(_workload(sys.argv[1])))
