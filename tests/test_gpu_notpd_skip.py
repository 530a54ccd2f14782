"""Pairs whose kernel matrix is not positive definite: once the diagonal block with the zero pivot has set the pair's
status, every later kernel of the blocked path returns for that pair at once.  The failing pairs must still report
what scikit-learn reports (-inf, zero gradient, _gpr.py:589-593), and the positive definite pairs of the same batch
must not change by a single bit."""
import numpy as np
import pytest
import scipy.linalg.lapack as lapack

import gp_oracle as orc

M = 1000                              # eight block columns of 128, the last one partial (104 rows)
FAIL_ROWS = (40, 434, 990)            # the zero pivot falls in block column 0, 3 and 7
TH_FAIL = np.log([1.0, 0.1, 1e-17])   # sigma^2 = 1, ell = 0.1, chi below half an ulp of 1
# positive definite thetas: a well-conditioned corner (cond(K) <= ~1e6 at m = 1000) of the eval_workload box
GOOD_LO, GOOD_HI = np.log([0.3, 0.01, 1e-2]), np.log([3.0, 0.1, 1e-1])


def _problem():
    """GP 0: synthetic trajectory.  GP 1 + k: abscissae 10 apart (with ell = 0.1 every off-diagonal kernel value
    underflows to exactly 0), except that row FAIL_ROWS[k] repeats the abscissa of the row before it.  With TH_FAIL the
    diagonal is exactly 1, so that row's pivot is exactly 1 - 1 * 1 = 0, in LAPACK and on the GPU alike."""
    t0, y = orc.synthetic_trajectories(1 + len(FAIL_ROWS), M, seed=3)
    T = np.empty((1 + len(FAIL_ROWS), M))
    T[0] = t0
    for k, r in enumerate(FAIL_ROWS):
        t = 10.0 * np.arange(M)
        t[r] = t[r - 1]
        T[1 + k] = t
    return T, y


def test_failing_rows_are_where_intended():
    T, _ = _problem()
    for k, r in enumerate(FAIL_ROWS):
        _, info = lapack.dpotrf(orc.np_kernel(T[1 + k], TH_FAIL), lower=1)
        assert info == r + 1, (k, info)                 # LAPACK's info is the 1-based row of the failed pivot


def _batches(B, seed):
    """Pair b fails (GP 1 + b % 3) when b % 2 == 1.  The reference batch replaces every failing pair by a positive
    definite one on GP 0: same size, so the same waves and split-K plans."""
    rng = np.random.default_rng(seed)
    theta_ref = rng.uniform(GOOD_LO, GOOD_HI, size=(B, 3))
    fail = np.arange(B) % 2 == 1
    theta = theta_ref.copy()
    theta[fail] = TH_FAIL
    gp_of = np.where(fail, 1 + np.arange(B) % len(FAIL_ROWS), 0).astype(np.int32)
    return theta, gp_of, theta_ref, np.zeros(B, dtype=np.int32), fail


def _check(lml, grad, st, ref, fail, with_grad):
    assert np.all(st[fail] == 1) and np.all(lml[fail] == -np.inf)
    ok = ~fail
    assert np.all(st[ok] == 0) and np.all(ref[2][ok] == 0)
    assert np.array_equal(lml[ok], ref[0][ok])
    if with_grad:
        assert np.all(grad[fail] == 0)
        assert np.array_equal(grad[ok], ref[1][ok])


# 12 pairs: the inverse rows run on the side stream (<= 148 pairs per wave); 200 pairs: everything on the main stream
@pytest.mark.gpu
@pytest.mark.parametrize("B", [12, 200])
def test_failed_pairs_skip_and_good_pairs_unchanged(ctx, B):
    T, y = _problem()
    theta, gp_of, theta_ref, gp_ref, fail = _batches(B, seed=B)
    for with_grad in (False, True):                   # with_grad=False: the LML-only path (block substitutions)
        got = ctx.lml_grad(T, y, theta, gp_of, with_grad=with_grad)
        ref = ctx.lml_grad(T, y, theta_ref, gp_ref, with_grad=with_grad)
        _check(*got, ref, fail, with_grad)
    lml, grad, _ = got
    for k in np.flatnonzero(~fail)[:3]:
        l0, g0, s0 = orc.np_lml_grad(T[0], y[0], theta[k])
        assert s0 == 0
        assert abs(lml[k] - l0) <= 1e-10 * abs(l0), (k, lml[k], l0)
        assert np.abs(grad[k] - g0).max() <= 1e-9 * max(1.0, np.abs(g0).max()), (k, grad[k], g0)


@pytest.mark.gpu
def test_failed_pairs_skip_over_several_waves(ctx):
    """A workspace that holds only a few pairs at m = 1000: failing and good pairs spread over several waves (the
    reference batch runs in the same waves; a one-wave run may differ in the last bits, its split-K plans differ)."""
    from gpbo_pkg import pkg

    T, y = _problem()
    B = 12
    theta, gp_of, theta_ref, gp_ref, fail = _batches(B, seed=7)
    small_ctx = pkg.Context(0, max_workspace_bytes=48 << 20)
    try:
        small_ctx.set_small_path(ctx.small_max)
        assert 1 < small_ctx.wave_capacity(M) < B
        got = small_ctx.lml_grad(T, y, theta, gp_of)
        ref = small_ctx.lml_grad(T, y, theta_ref, gp_ref)
    finally:
        small_ctx.close()
    _check(*got, ref, fail, True)
