"""ctypes binding of ``libgpbo.so`` (C ABI declared in ``include/gpbo.h``).

This is the whole host<->device boundary of the package: plain pointers and sizes, no torch
types.  There is NO CPU fallback -- if the shared library is missing or no CUDA device is
present, every compute call raises.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# GPBO_LIB: an alternative build of the same library (A/B measurements of kernel variants, tools/ab/); never a fallback
LIB_PATH = os.environ.get("GPBO_LIB") or os.path.join(_HERE, "libgpbo.so")

NCLASS = 14
KERNEL_CLASSES = ("prep", "chol_diag", "chol_panel", "trsv", "trtri", "lauum_grad", "finalize",
                  "cross_panel", "schur", "mean_std", "assemble", "sqrtw", "small", "std")

OBJECTIVE_FN = C.CFUNCTYPE(C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p)

_I, _L, _D, _V = C.c_int, C.c_long, C.c_double, C.c_void_p
_PD, _PI, _PLL, _PV = C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_longlong), C.POINTER(C.c_void_p)
# entry point of include/gpbo.h -> (restype, argtypes)
_SIGNATURES = {
    "gpbo_version": (_I, []),
    "gpbo_last_error": (C.c_char_p, []),
    "gpbo_create": (_I, [_PV, _I, C.c_size_t]),
    "gpbo_destroy": (_I, [_V]),
    "gpbo_launch_count": (C.c_longlong, [_V]),
    "gpbo_wave_capacity": (_I, [_V, _I]),
    "gpbo_set_kernel_family": (_I, [_V, _I]),
    "gpbo_assemble": (_I, [_V, _I, _V, _L, _I, _V, _L, _I, _V, _I, _V, _V]),
    "gpbo_assemble_matern": (_I, [_V, _I, _I, _V, _L, _I, _V, _L, _I, _V, _I, _V, _V]),
    "gpbo_lml_grad": (_I, [_V, _V, _V, _I, _I, _V, _V, _I, _V, _V, _V, _V]),
    "gpbo_lml_grad_host": (_I, [_V, _PD, _PD, _I, _I, _PD, _PI, _I, _PD, _PD, _PI]),
    "gpbo_fit_host": (_I, [_V, _PD, _PD, _I, _I, _PD, _PD, _PI, _I, _PD, _PD, _PD, _PI, _PI, _PI, _PLL, _PI]),
    "gpbo_predict_host": (_I, [_V, _PD, _PD, _I, _I, _PD, _PD, _L, _I, _PD, _PD, _PD, _PI]),
    "gpbo_lstsq_moments_host": (_I, [_V, _PD, _PD, _I, _I, _PD, _PD, _L, _I, _PD, _PD, _PD, _PI]),
    "gpbo_lstsq_moments": (_I, [_V, _V, _V, _I, _I, _V, _V, _L, _I, _V, _V, _V, _V, _V]),
    "gpbo_sqrtw": (_I, [_V, _V, _I, _I, _D, _V, _PI, _PI, _V]),
    "gpbo_sqrtw_host": (_I, [_V, _PD, _I, _I, _D, _PD, _PI, _PI]),
    "gpbo_lstsq_weights_host": (_I, [_V, _PD, _PD, _I, _I, _PD, _PD, _L, _I, _D, _PD, _PD, _PD, _PD, _PI, _PI, _PI]),
    "gpbo_weighted_products_host": (_I, [_V, _PD, _I, _I, _PD, _I, _PD, _PD, _PD]),
    "gpbo_posterior_grid_host": (_I, [_V, _PD, _I, _I, _PD, _I, _PD, _PD, _I, _PD, _PD, _PD, _PD, _PI]),
    "gpbo_set_small_path": (_I, [_V, _I]),
    "gpbo_get_stream": (_I, [_V, _PV]),
    "gpbo_optpool_create": (_I, [_PV, _I, _PD, _PD, _PD]),
    "gpbo_optpool_destroy": (_I, [_V]),
    "gpbo_optpool_live": (_I, [_V, _PI, _PD, _PI]),
    "gpbo_optpool_feed": (_I, [_V, _I, _PI, _PD, _PD]),
    "gpbo_optpool_result": (_I, [_V, _PD, _PD, _PI, _PI, _PI, _PLL, _PI]),
    "gpbo_problem_upload_host": (_I, [_V, _PD, _PD, _I, _I]),
    "gpbo_lml_grad_resident_host": (_I, [_V, _PD, _PI, _I, _PD, _PD, _PI]),
    "gpbo_profile_enable": (_I, [_V, _I]),
    "gpbo_profile_get": (_I, [_V, _PD, _PLL]),
    "gpbo_bench_dmma_peak": (_I, [_V, _I, _PD, _PD]),
    "gpbo_lbfgsb_minimize": (_I, [OBJECTIVE_FN, _V, _PD, _PD, _PD, _PD, _PD, _PI, _PI, _PI]),
}
EXPORTS = tuple(_SIGNATURES)


class GpboError(RuntimeError):
    """Raised when a libgpbo call returns a non-zero status."""


_lib = None


def load():
    """Load libgpbo.so (built by ``__graft_entry__.build()`` / ``csrc/Makefile``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise GpboError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = lib
    return lib


def _check(rc, what):
    if rc != 0:
        msg = load().gpbo_last_error().decode("utf-8", "replace")
        raise GpboError(f"{what} failed (status {rc}): {msg}")


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int))


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _problem(t, y, theta=None, n_theta=None):
    """Validate the (t, y[, theta]) arguments the way scikit-learn validates X / y (``ValueError`` on inconsistent
    numbers of samples) -- the C side reads G*m doubles from each of t and y and 3 per theta row."""
    t, y = _f64(np.atleast_2d(t)), _f64(np.atleast_2d(y))
    if t.ndim != 2 or y.shape != t.shape:
        raise ValueError(f"Found input variables with inconsistent numbers of samples: t {t.shape}, y {y.shape}")
    if t.shape[1] == 0:
        raise ValueError("at least one training sample is required")
    if theta is None:
        return t, y
    theta = _f64(np.atleast_2d(theta))
    if theta.ndim != 2 or theta.shape[1] != 3 or (n_theta is not None and theta.shape[0] != n_theta):
        want = "(B, 3)" if n_theta is None else f"({n_theta}, 3)"
        raise ValueError(f"theta must have shape {want}, got {theta.shape}")
    return t, y, theta


def _gp_of(gp_of, B, G):
    if gp_of is None:
        if B != G:
            raise ValueError(f"gp_of is required when the number of pairs ({B}) differs from the number of GPs ({G})")
        return None
    gp = np.ascontiguousarray(gp_of, dtype=np.int32)
    if gp.shape != (B,):
        raise ValueError(f"gp_of must have shape ({B},), got {gp.shape}")
    if gp.size and (gp.min() < 0 or gp.max() >= G):
        raise ValueError("gp_of entry out of range")
    return gp


def _step3_operands(lhs, rhs, sqrtW):
    """lhs (n, d), rhs (G, n) and sqrtW (G, n, n) or None of the step-3 products, as contiguous float64 arrays with
    consistent shapes."""
    lhs = _f64(lhs)
    rhs = _f64(np.atleast_2d(rhs))
    G, n = rhs.shape
    if lhs.ndim != 2 or lhs.shape[0] != n:
        raise ValueError(f"expected lhs.shape == ({n}, d)")
    w = None
    if sqrtW is not None:
        w = _f64(sqrtW)
        if w.shape != (G, n, n):
            raise ValueError(f"expected sqrtW.shape == ({G}, {n}, {n})")
    return lhs, rhs, w


class OptimizerPool:
    """The B L-BFGS-B state machines of a multi-start fit (``gpbo_optpool_*``; host memory only).  ``live()`` gives
    the running pairs and their trial points, ``feed()`` takes their LML / gradient -- the loop of
    ``gpbo_fit_host`` opened up so that ``sharding.fit_pairs`` can all-gather between the two."""

    def __init__(self, bounds_log, starts, opts=None):
        self._lib = load()
        starts = _f64(np.atleast_2d(starts))
        if starts.ndim != 2 or starts.shape[1] != 3:
            raise ValueError("starts must have shape (B, 3)")
        self.B = starts.shape[0]
        bl = _f64(bounds_log, (3, 2))
        o = None if opts is None else _f64(opts, (5,))
        h = C.c_void_p()
        _check(self._lib.gpbo_optpool_create(C.byref(h), self.B, _dp(bl), _dp(starts), _dp(o)), "gpbo_optpool_create")
        self._h = h
        self._idx = np.empty(self.B, dtype=np.int32)
        self._theta = np.empty((self.B, 3))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gpbo_optpool_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def live(self):
        """-> (idx (n,) int32, theta (n, 3)) of the optimisers that still run (copies)."""
        n = C.c_int()
        _check(self._lib.gpbo_optpool_live(self._h, _ip(self._idx), _dp(self._theta), C.byref(n)), "gpbo_optpool_live")
        return self._idx[:n.value].copy(), self._theta[:n.value].copy()

    def feed(self, idx, lml, grad):
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        lml = _f64(lml)
        grad = _f64(grad)
        if lml.shape != idx.shape or grad.shape != (idx.size, 3):
            raise ValueError("feed: shape mismatch")
        _check(self._lib.gpbo_optpool_feed(self._h, int(idx.size), _ip(idx), _dp(lml), _dp(grad)), "gpbo_optpool_feed")

    def result(self):
        B = self.B
        theta, fun = np.empty((B, 3)), np.empty(B)
        nfev, nit, st = (np.empty(B, dtype=np.int32) for _ in range(3))
        evals, rounds = C.c_longlong(), C.c_int()
        _check(self._lib.gpbo_optpool_result(self._h, _dp(theta), _dp(fun), _ip(nfev), _ip(nit), _ip(st),
                                             C.byref(evals), C.byref(rounds)), "gpbo_optpool_result")
        return dict(theta=theta, fun=fun, nfev=nfev, nit=nit, status=st, evals=int(evals.value),
                    rounds=int(rounds.value))


class Context:
    """Owns one ``gpbo_ctx`` workspace handle on a CUDA device."""

    def __init__(self, device: int = 0, max_workspace_bytes: int = 0):
        self._lib = load()
        h = C.c_void_p()
        _check(self._lib.gpbo_create(C.byref(h), int(device), int(max_workspace_bytes)), "gpbo_create")
        self._h = h
        self.device = int(device)
        self.small_max = 224          # sizes up to this run on the in-shared small-matrix path (set_small_path)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gpbo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- bookkeeping -----------------------------------------------------------------
    @property
    def launch_count(self) -> int:
        return int(self._lib.gpbo_launch_count(self._h))

    def set_kernel_family(self, twice_nu: int = 0):
        """0: RBF (the reference); 3 / 5: Matern nu = 3/2, 5/2.  Applies to all later calls on this context."""
        _check(self._lib.gpbo_set_kernel_family(self._h, int(twice_nu)), "gpbo_set_kernel_family")

    @property
    def stream(self) -> int:
        """Address of the cudaStream_t the host-pointer entry points run on."""
        p = C.c_void_p()
        _check(self._lib.gpbo_get_stream(self._h, C.byref(p)), "gpbo_get_stream")
        return int(p.value or 0)

    def set_small_path(self, max_m: int = 224):
        """Training sizes m <= max_m use the in-shared one-launch path (default 224); 0: always the blocked path."""
        _check(self._lib.gpbo_set_small_path(self._h, int(max_m)), "gpbo_set_small_path")
        self.small_max = min(int(max_m), 224)

    def upload_problem(self, t, y):
        """Keep (t, y): (G, m) resident in HBM for ``lml_grad_resident``."""
        t, y = _problem(t, y)
        _check(self._lib.gpbo_problem_upload_host(self._h, _dp(t), _dp(y), t.shape[0], t.shape[1]),
               "gpbo_problem_upload_host")
        self._resident = t.shape

    def lml_grad_resident(self, theta, gp_of):
        """LML + gradient of B pairs against the resident problem.  -> lml (B,), grad (B, 3), status (B,)."""
        theta = _f64(np.atleast_2d(theta))
        B = theta.shape[0]
        if theta.ndim != 2 or (B and theta.shape[1] != 3):
            raise ValueError("theta must have shape (B, 3)")
        lml, grad, st = np.empty(B), np.empty((B, 3)), np.empty(B, dtype=np.int32)
        if B == 0:
            return lml, grad, st
        if gp_of is None or getattr(self, "_resident", None) is None:
            raise ValueError("lml_grad_resident needs gp_of and a problem uploaded with upload_problem()")
        gp = _gp_of(gp_of, B, self._resident[0])
        _check(self._lib.gpbo_lml_grad_resident_host(self._h, _dp(theta), _ip(gp), B, _dp(lml), _dp(grad), _ip(st)),
               "gpbo_lml_grad_resident_host")
        return lml, grad, st

    def wave_capacity(self, m: int) -> int:
        return int(self._lib.gpbo_wave_capacity(self._h, int(m)))

    def profile_enable(self, on=True):
        _check(self._lib.gpbo_profile_enable(self._h, 1 if on else 0), "gpbo_profile_enable")

    def profile_get(self):
        ms = np.zeros(NCLASS)
        n = np.zeros(NCLASS, dtype=np.int64)
        _check(self._lib.gpbo_profile_get(self._h, _dp(ms), n.ctypes.data_as(C.POINTER(C.c_longlong))),
               "gpbo_profile_get")
        return {k: (float(ms[i]), int(n[i])) for i, k in enumerate(KERNEL_CLASSES)}

    def dmma_peak(self, iters=20000):
        tf, ms = C.c_double(), C.c_double()
        _check(self._lib.gpbo_bench_dmma_peak(self._h, int(iters), C.byref(tf), C.byref(ms)), "gpbo_bench_dmma_peak")
        return tf.value, ms.value

    # -- host-pointer entry points ------------------------------------------------------
    def lml_grad(self, t, y, theta, gp_of=None, with_grad=True):
        """t, y: (G, m); theta: (B, 3); gp_of: (B,) int or None (B == G). -> lml (B,), grad (B,3), status (B,)."""
        t, y, theta = _problem(t, y, theta)
        G, m = t.shape
        B = theta.shape[0]
        gp = _gp_of(gp_of, B, G)
        lml = np.empty(B)
        grad = np.empty((B, 3)) if with_grad else None
        st = np.empty(B, dtype=np.int32)
        _check(self._lib.gpbo_lml_grad_host(self._h, _dp(t), _dp(y), G, m, _dp(theta), _ip(gp), B, _dp(lml),
                                            _dp(grad), _ip(st)), "gpbo_lml_grad_host")
        return lml, grad, st

    def fit(self, t, y, bounds_log, starts, gp_of=None, opts=None):
        """Multi-start L-BFGS-B for all (GP, start) pairs in lock-step.

        bounds_log: (3, 2); starts: (B, 3).  Returns dict(theta, fun, nfev, nit, status, evals, rounds)."""
        t, y, starts = _problem(t, y, starts)
        G, m = t.shape
        B = starts.shape[0]
        bl = _f64(bounds_log, (3, 2))
        gp = _gp_of(gp_of, B, G)
        o = None if opts is None else _f64(opts, (5,))
        theta = np.empty((B, 3))
        fun = np.empty(B)
        nfev = np.empty(B, dtype=np.int32)
        nit = np.empty(B, dtype=np.int32)
        st = np.empty(B, dtype=np.int32)
        evals = C.c_longlong()
        rounds = C.c_int()
        _check(self._lib.gpbo_fit_host(self._h, _dp(t), _dp(y), G, m, _dp(bl), _dp(starts), _ip(gp), B, _dp(o),
                                       _dp(theta), _dp(fun), _ip(nfev), _ip(nit), _ip(st), C.byref(evals),
                                       C.byref(rounds)), "gpbo_fit_host")
        return dict(theta=theta, fun=fun, nfev=nfev, nit=nit, status=st, evals=int(evals.value),
                    rounds=int(rounds.value))

    def _points(self, pts, G):
        pts = _f64(pts)
        if pts.ndim == 1:
            if pts.shape[0] == 0:
                raise ValueError("at least one evaluation point is required")
            return pts, 0, pts.shape[0]
        if pts.ndim != 2 or pts.shape[0] != G or pts.shape[1] == 0:
            raise ValueError("per-GP evaluation points must have shape (G, n)")
        return pts, pts.shape[1], pts.shape[1]

    def predict(self, t, y, theta, t_star, want_alpha=False):
        """Posterior mean and std at t_star ((n,) shared or (G, n)).  -> mean, std, alpha|None, status."""
        t, y, theta = _problem(t, y, theta, n_theta=np.atleast_2d(t).shape[0])
        G, m = t.shape
        pts, stride, n = self._points(t_star, G)
        mean, std = np.empty((G, n)), np.empty((G, n))
        alpha = np.empty((G, m)) if want_alpha else None
        st = np.empty(G, dtype=np.int32)
        _check(self._lib.gpbo_predict_host(self._h, _dp(t), _dp(y), G, m, _dp(theta), _dp(pts), stride, n, _dp(mean),
                                           _dp(std), _dp(alpha), _ip(st)), "gpbo_predict_host")
        return mean, std, alpha, st

    def lstsq_moments(self, t, y, theta, t_est, want_cov=True):
        """state_estimate, ddt_estimate, ddt_covariance at t_est.  -> state, ddt, cov|None, status."""
        t, y, theta = _problem(t, y, theta, n_theta=np.atleast_2d(t).shape[0])
        G, m = t.shape
        pts, stride, n = self._points(t_est, G)
        state, ddt = np.empty((G, n)), np.empty((G, n))
        cov = np.empty((G, n, n)) if want_cov else None
        st = np.empty(G, dtype=np.int32)
        _check(self._lib.gpbo_lstsq_moments_host(self._h, _dp(t), _dp(y), G, m, _dp(theta), _dp(pts), stride, n,
                                                 _dp(state), _dp(ddt), _dp(cov), _ip(st)), "gpbo_lstsq_moments_host")
        return state, ddt, cov, st

    def sqrtw(self, cov, eta):
        """sqrtW = (C + eta I)^(-1/2) for a stack of covariances (G, n, n).  -> sqrtw, status, iters."""
        cov = _f64(cov)
        if cov.ndim == 2:
            cov = cov[None]
        G, n, n2 = cov.shape
        if n != n2:
            raise ValueError("sqrtw: covariance must be square")
        out = np.empty_like(cov)
        st = np.empty(G, dtype=np.int32)
        it = np.empty(G, dtype=np.int32)
        _check(self._lib.gpbo_sqrtw_host(self._h, _dp(cov), G, n, float(eta), _dp(out), _ip(st), _ip(it)),
               "gpbo_sqrtw_host")
        return out, st, it

    def lstsq_weights(self, t, y, theta, t_est, eta):
        """state, ddt, cov AND sqrtW in one call (the covariance never leaves HBM in between).
        -> state, ddt, cov, sqrtw, status, w_status, w_iters."""
        t, y, theta = _problem(t, y, theta, n_theta=np.atleast_2d(t).shape[0])
        G, m = t.shape
        pts, stride, n = self._points(t_est, G)
        state, ddt = np.empty((G, n)), np.empty((G, n))
        cov, w = np.empty((G, n, n)), np.empty((G, n, n))
        st, wst, wit = (np.empty(G, dtype=np.int32) for _ in range(3))
        _check(self._lib.gpbo_lstsq_weights_host(self._h, _dp(t), _dp(y), G, m, _dp(theta), _dp(pts), stride, n,
                                                 float(eta), _dp(state), _dp(ddt), _dp(cov), _dp(w), _ip(st), _ip(wst),
                                                 _ip(wit)), "gpbo_lstsq_weights_host")
        return state, ddt, cov, w, st, wst, wit

    def weighted_products(self, lhs, rhs, sqrtW=None):
        """(sqrtW[g] @ lhs, sqrtW[g] @ rhs[g]) for all g (wlstsq.py:183-188).  sqrtW=None: use the weight matrices
        resident on the device since the last lstsq_weights / sqrtw call (same G, n).  -> (G, n, d), (G, n)."""
        lhs, rhs, w = _step3_operands(lhs, rhs, sqrtW)
        (G, n), d = rhs.shape, lhs.shape[1]
        out_lhs, out_rhs = np.empty((G, n, d)), np.empty((G, n))
        _check(self._lib.gpbo_weighted_products_host(self._h, _dp(w), G, n, _dp(lhs), d, _dp(rhs), _dp(out_lhs),
                                                     _dp(out_rhs)), "gpbo_weighted_products_host")
        return out_lhs, out_rhs

    def posterior_grid(self, lhs, rhs, regularizers, sqrtW=None, want_chol=True):
        """Step-3 posterior assembly for a grid of regularizers (PDEs/step3_estimate.py:75-95 for every candidate of
        :131-148): per GP g and regularizer k the posterior mean of the operator row, the Cholesky factor of its
        precision ``(sqrtW_g D)^T (sqrtW_g D) + reg_k^2 I`` and whether that precision is positive definite.
        sqrtW=None: the weight matrices resident on the device since the last lstsq_weights / sqrtw call.
        -> dict(means (K, G, d), chol (K, G, d, d) | None, gram (G, d, d), proj (G, d), status (K, G))."""
        lhs, rhs, w = _step3_operands(lhs, rhs, sqrtW)
        (G, n), d = rhs.shape, lhs.shape[1]
        regs = _f64(np.atleast_1d(regularizers))
        if regs.ndim != 1 or regs.size == 0 or not np.all(np.isfinite(regs)):
            raise ValueError("regularizers must be a non-empty 1-D array of finite values")
        K = regs.size
        means = np.empty((K, G, d))
        chol = np.empty((K, G, d, d)) if want_chol else None
        gram, proj = np.empty((G, d, d)), np.empty((G, d))
        status = np.empty((K, G), dtype=np.int32)
        _check(self._lib.gpbo_posterior_grid_host(self._h, _dp(w), G, n, _dp(lhs), d, _dp(rhs), _dp(regs), K, _dp(means),
                                                  _dp(chol), _dp(gram), _dp(proj), _ip(status)),
               "gpbo_posterior_grid_host")
        return {"means": means, "chol": chol, "gram": gram, "proj": proj, "status": status}

    # -- device-pointer entry points (torch tensors are only address carriers) ------------
    def assemble_device(self, kind, t1_ptr, t1_stride, n1, t2_ptr, t2_stride, n2, theta_ptr, B, out_ptr, stream=0,
                        twice_nu=0):
        """twice_nu = 0: RBF (gpbo_assemble); 3 / 5: Matern nu = 3/2, 5/2 (gpbo_assemble_matern)."""
        if twice_nu:
            _check(self._lib.gpbo_assemble_matern(self._h, int(twice_nu), int(kind), t1_ptr, int(t1_stride), int(n1),
                                                  t2_ptr, int(t2_stride), int(n2), theta_ptr, int(B), out_ptr, stream),
                   "gpbo_assemble_matern")
            return
        _check(self._lib.gpbo_assemble(self._h, int(kind), t1_ptr, int(t1_stride), int(n1), t2_ptr, int(t2_stride),
                                       int(n2), theta_ptr, int(B), out_ptr, stream), "gpbo_assemble")

    def lml_grad_device(self, t_ptr, y_ptr, G, m, theta_ptr, gpof_ptr, B, lml_ptr, grad_ptr, status_ptr, stream=0):
        _check(self._lib.gpbo_lml_grad(self._h, t_ptr, y_ptr, int(G), int(m), theta_ptr, gpof_ptr, int(B), lml_ptr,
                                       grad_ptr, status_ptr, stream), "gpbo_lml_grad")

    def lstsq_moments_device(self, t_ptr, y_ptr, G, m, theta_ptr, test_ptr, test_stride, n, state_ptr, ddt_ptr,
                             cov_ptr, status_ptr, stream=0):
        _check(self._lib.gpbo_lstsq_moments(self._h, t_ptr, y_ptr, int(G), int(m), theta_ptr, test_ptr,
                                            int(test_stride), int(n), state_ptr, ddt_ptr, cov_ptr, status_ptr, stream),
               "gpbo_lstsq_moments")


_default_ctx = {}


def default_context(device: int | None = None) -> Context:
    """Process-wide context for `device` (default: LOCAL_RANK or 0)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


def lbfgsb_minimize(func, x0, bounds_log, opts=None):
    """Host-only run of the library's L-BFGS-B state machine on ``func(x) -> (f, g)`` (3 variables).
    No CUDA device needed; used by the CPU tests to pin the optimiser against scipy."""
    lib = load()

    def _cb(xp, gp, _user):
        x = np.array([xp[0], xp[1], xp[2]])
        f, g = func(x)
        for i in range(3):
            gp[i] = float(g[i])
        return float(f)

    cb = OBJECTIVE_FN(_cb)
    x0 = _f64(x0, (3,))
    bl = _f64(bounds_log, (3, 2))
    o = None if opts is None else _f64(opts, (5,))
    x = np.empty(3)
    f = C.c_double()
    nfev, nit, st = C.c_int(), C.c_int(), C.c_int()
    _check(lib.gpbo_lbfgsb_minimize(cb, None, _dp(x0), _dp(bl), _dp(o), _dp(x), C.byref(f), C.byref(nfev),
                                    C.byref(nit), C.byref(st)), "gpbo_lbfgsb_minimize")
    return dict(x=x, fun=f.value, nfev=nfev.value, nit=nit.value, status=st.value)
