"""Import the UNMODIFIED reference (``/root/reference``) in the build container.

TEST INFRASTRUCTURE ONLY (see ``oracle/gp_oracle.py``).  ``/root/reference``
does not exist on the GPU box, so nothing in ``-m gpu`` tests, ``smoke()`` or
``bench.py`` may import this module; it is used by ``oracle/make_golden.py`` to
write ``tests/golden/*.npz``; the tests compare with what it stored there and
never import the reference themselves.

The reference needs packages that are not installed here (gpytorch, opinf,
matplotlib, IPython).  Only the exact names the reference touches at import
time are stubbed (SURVEY.md §8c, Appendix A); no reference source is copied.
"""

from __future__ import annotations

import contextlib
import importlib
import os
import sys
import time
import types

REFERENCE_ROOT = os.environ.get("GPBO_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "codebase", "gpkernels.py"))


def _mk(name, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


class _Dummy:
    def __init__(self, *a, **k):
        pass


class _TimedBlock(contextlib.ContextDecorator):
    """Stand-in for opinf.utils.TimedBlock (wall-clock print wrapper)."""

    def __init__(self, message="", timelimit=None):
        self.message = message

    def __enter__(self):
        self.t0 = time.time()
        return self

    def __exit__(self, *exc):
        return False


def install_stubs():
    """Stub gpytorch / opinf.utils / matplotlib / IPython (names used at import time only)."""
    try:
        import gpytorch  # noqa: F401
    except Exception:
        _mk("gpytorch")
        _mk("gpytorch.models", ExactGP=_Dummy)
        _mk("gpytorch.likelihoods", GaussianLikelihood=_Dummy)
        _mk("gpytorch.means", ZeroMean=_Dummy)
        _mk("gpytorch.kernels", ScaleKernel=_Dummy, RBFKernel=_Dummy)
    try:
        import opinf  # noqa: F401
    except Exception:
        op = _mk("opinf")
        op.utils = _mk("opinf.utils", TimedBlock=_TimedBlock)
    try:
        import matplotlib  # noqa: F401
    except Exception:
        mpl = _mk("matplotlib")
        for sub in ("pyplot", "colors", "animation", "patches"):
            setattr(mpl, sub, _mk(f"matplotlib.{sub}"))
    try:
        import IPython  # noqa: F401
    except Exception:
        ip = _mk("IPython")
        ip.display = _mk("IPython.display", HTML=_Dummy)


def load_reference_gpkernels():
    """Return the reference's ``codebase/gpkernels.py`` module (sklearn path = the oracle)."""
    if not reference_available():
        raise FileNotFoundError(f"reference not found under {REFERENCE_ROOT}")
    install_stubs()
    path = os.path.join(REFERENCE_ROOT, "codebase")
    if path not in sys.path:
        sys.path.insert(0, path)
    mod = importlib.import_module("gpkernels")
    if not os.path.realpath(mod.__file__).startswith(os.path.realpath(REFERENCE_ROOT)):
        raise ImportError(f"'gpkernels' resolved to {mod.__file__}, not the reference")
    return mod


def load_reference_models():
    """Return (ode_models, pde_models) from the reference's ``models/`` directory."""
    install_stubs()
    path = os.path.join(REFERENCE_ROOT, "models")
    if path not in sys.path:
        sys.path.insert(0, path)
    return importlib.import_module("ode_models"), importlib.import_module("pde_models")
