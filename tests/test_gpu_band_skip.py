"""Short length scales: with ell far below the spread of t, whole 128 x 128 tiles of the RBF kernel matrix are exactly
zero, and the blocked path skips them (the factor's profile in chol_diag / chol_panel / the split-K partials, the
profile of the inverse rows in trtri_row, the tiles outside the band in lauum_grad).  The abscissae are unsorted but
block-local (the sorted grid's 128-point runs in shuffled order, each run shuffled), so the rule still finds zero tiles;
every test first checks with the numpy restatement of the rule (tools/ab_bench.py, band_profile) that its short-ell
pairs really take the shortened loops.  The batches mix such pairs with dense ones, with a pair that is not positive
definite, over one and several waves; small batches go through the split-K partials and the side stream, a batch of
160 pairs at m = 2048 runs most block columns and rows with their own k-loops.  LML and gradient are checked against
the dense LAPACK oracle at the bars of the rest of the suite, LML-only calls included."""
import os
import sys

import numpy as np
import pytest

import gp_oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from ab_bench import band_profile  # noqa: E402

SHORT = np.log([[0.3, 1e-4, 1e-2], [3.0, 5e-3, 1e-1]])    # sigma^2, ell, chi: banded K
DENSE = np.log([[0.3, 0.05, 1e-2], [3.0, 0.3, 1e-1]])     # well conditioned, dense K
TH_FAIL = np.log([1.0, 0.1, 1e-17])                       # with GP 1 below: a zero pivot in block column 3
TB = 128


@pytest.fixture(scope="module")
def bctx():
    from gpbo_pkg import pkg

    c = pkg.Context(0)
    c.set_kernel_family(0)
    c.set_small_path(0)
    yield c
    c.close()


def _block_local_perm(m, rng):
    """The full 128-point runs of 0..m-1 in shuffled order, each shuffled; a partial last run stays last."""
    full = m // TB
    runs = [rng.permutation(np.arange(b * TB, (b + 1) * TB)) for b in rng.permutation(full)]
    if m % TB:
        runs.append(rng.permutation(np.arange(full * TB, m)))
    return np.concatenate(runs)


def _problem(m, seed):
    """GP 0: a synthetic trajectory with its points in block-local random order (the kernels do not assume sorted t).
    GP 1: t 10 apart, with row 434 repeating the abscissa before it -- under TH_FAIL every off-diagonal element is
    exactly 0 and that pivot is exactly 0."""
    t, y = orc.synthetic_trajectories(2, m, seed=seed)
    perm = _block_local_perm(m, np.random.default_rng(seed))
    T = np.empty((2, m))
    T[0] = t[perm]
    y = y[:, perm].copy()
    T[1] = 10.0 * np.arange(m)
    T[1, 434] = T[1, 433]
    return T, y


def _thetas(B, seed):
    rng = np.random.default_rng(seed)
    short = rng.uniform(0, 1, size=B) < 0.6
    lo = np.where(short[:, None], SHORT[0], DENSE[0])
    hi = np.where(short[:, None], SHORT[1], DENSE[1])
    theta = lo + (hi - lo) * rng.uniform(size=(B, 3))
    theta[0, 1] = np.log(1e-4)
    theta[1, 1] = np.log(2e-3)
    return theta


def _assert_skips(t, theta, m):
    """The batch holds pairs whose loops the profile shortens but does not empty: a panel tile (i, j) with
    0 < max(f(i), f(j)) < j, an inverse tile with f(i) > j (dense first block), a lauum tile outside the band."""
    panel = trtri = lauum = False
    for th in theta:
        zero, f = band_profile(t, np.exp(th[1]), m)
        T = len(f)
        for i in range(T):
            for j in range(i):
                kb = max(f[i], f[j])
                panel |= j >= f[i] and 0 < kb < j
                trtri |= j < f[i] < i
                lauum |= bool(zero[i, j])
    assert panel and trtri and lauum


def _check_oracle(T, y, theta, gp_of, lml, grad, st, with_grad, n_check):
    bad = np.flatnonzero(gp_of == 1)
    assert np.all(st[bad] == 1) and np.all(lml[bad] == -np.inf)
    if with_grad:
        assert np.all(grad[bad] == 0)
    good = np.flatnonzero(gp_of == 0)
    assert np.all(st[good] == 0)
    # the shortest length scales first: those are the pairs that skip the most; then the longest as a dense control
    order = good[np.argsort(theta[good, 1])]
    for b in np.concatenate([order[:n_check], order[-1:]]):
        l0, g0, s0 = orc.np_lml_grad_lean(T[0], y[0], theta[b])
        assert s0 == 0
        assert abs(lml[b] - l0) <= 1e-10 * abs(l0), (b, theta[b], lml[b], l0)
        if with_grad:
            assert np.abs(grad[b] - g0).max() <= 1e-9 * max(1.0, np.abs(g0).max()), (b, theta[b], grad[b], g0)


# B = 3: split-K partials and the inverse rows on the side stream; B = 40: side stream; B = 200 (m = 1000) and
# B = 160 (m = 2048): main stream, most block columns and rows without split-K
@pytest.mark.gpu
@pytest.mark.parametrize("m,B", [(1000, 3), (1000, 200), (2048, 3), (2048, 40), (2048, 160)])
def test_banded_batches_match_oracle(bctx, m, B):
    T, y = _problem(m, seed=m + B)
    theta = _thetas(B, seed=B)
    gp_of = np.zeros(B, dtype=np.int32)
    if B > 3:
        theta[B // 2] = TH_FAIL
        gp_of[B // 2] = 1
    _assert_skips(T[0], theta[gp_of == 0], m)
    for with_grad in (True, False):                  # with_grad=False: the LML-only path (block substitutions)
        lml, grad, st = bctx.lml_grad(T, y, theta, gp_of, with_grad=with_grad)
        _check_oracle(T, y, theta, gp_of, lml, grad, st, with_grad, n_check=3)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [24, 160])
def test_replicated_pairs_bit_identical(bctx, B):
    """Copies of one pair in one batch take the same skips and give the same bits, whatever their position; with
    B = 160 the copies run the unsplit k-loops.  LML-only as well."""
    m = 2048
    T, y = _problem(m, seed=5)
    base = _thetas(8, seed=9)
    _assert_skips(T[0], base, m)
    theta = np.tile(base, (B // 8, 1))
    gp_of = np.zeros(B, dtype=np.int32)
    for with_grad in (True, False):
        lml, grad, st = bctx.lml_grad(T, y, theta, gp_of, with_grad=with_grad)
        assert np.all(st == 0)
        for k in range(8):
            assert np.all(lml[k::8] == lml[k]), (with_grad, k)
            if with_grad:
                assert np.all(grad[k::8] == grad[k]), k


@pytest.mark.gpu
def test_banded_pairs_over_several_waves():
    """A workspace that holds only a few pairs at m = 1000: banded, dense and failing pairs spread over several
    waves."""
    from gpbo_pkg import pkg

    m, B = 1000, 12
    T, y = _problem(m, seed=17)
    theta = _thetas(B, seed=4)
    gp_of = np.zeros(B, dtype=np.int32)
    theta[7] = TH_FAIL
    gp_of[7] = 1
    _assert_skips(T[0], theta[gp_of == 0], m)
    c = pkg.Context(0, max_workspace_bytes=48 << 20)
    try:
        c.set_kernel_family(0)
        c.set_small_path(0)
        assert 1 < c.wave_capacity(m) < B
        lml, grad, st = c.lml_grad(T, y, theta, gp_of)
    finally:
        c.close()
    _check_oracle(T, y, theta, gp_of, lml, grad, st, True, n_check=3)


@pytest.mark.gpu
def test_all_off_diagonal_tiles_zero(bctx):
    """ell = 1e-4 at m = 2048 on sorted t: nearly every tile off the diagonal is exactly zero, so the factor is
    close to block diagonal and the inverse rows and gradient tiles are almost all skipped.  LML and gradient
    against the dense computation on the CPU."""
    m = 2048
    t, y = orc.synthetic_trajectories(1, m, seed=23)
    theta = np.log([[1.7, 1e-4, 3e-2], [0.4, 2e-3, 1e-2]])
    _assert_skips(t, theta, m)
    lml, grad, st = bctx.lml_grad(t[None, :], y, theta, np.zeros(2, dtype=np.int32))
    for b in range(2):
        l0, g0, s0 = orc.np_lml_grad(t, y[0], theta[b])
        assert st[b] == 0 and s0 == 0
        assert abs(lml[b] - l0) <= 1e-10 * abs(l0), (b, lml[b], l0)
        assert np.abs(grad[b] - g0).max() <= 1e-9 * max(1.0, np.abs(g0).max()), (b, grad[b], g0)
