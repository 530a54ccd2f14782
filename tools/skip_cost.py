"""What a CTA costs that returns at once because its pair's Cholesky already failed (pair_failed() in kernels_chol.cuh).

    python tools/skip_cost.py [m] [pairs]

Every pair of one wave fails at row 1 (block column 0): abscissae 10 apart, the first two equal, sigma^2 = 1, ell = 0.1,
chi = 1e-17, so the pivot of row 1 is exactly 0.  Each kernel class then runs its full grid of CTAs that all return at
once (except chol_diag for j = 0).  Prints the CUDA-event time per class and per CTA as one JSON line.
"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gpbo_pkg import pkg  # noqa: E402

m = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
B = int(sys.argv[2]) if len(sys.argv) > 2 else 256
REPS = 3
t = 10.0 * np.arange(m)
t[1] = t[0]
theta = np.tile(np.log([1.0, 0.1, 1e-17]), (B, 1))
gp_of = np.zeros(B, dtype=np.int32)
ctx = pkg.default_context(0)
ctx.upload_problem(t[None], np.zeros((1, m)))
assert ctx.wave_capacity(m) >= B
_, _, st = ctx.lml_grad_resident(theta, gp_of)
assert np.all(st == 1)
ctx.profile_enable(True)
for _ in range(REPS):
    ctx.lml_grad_resident(theta, gp_of)
prof = ctx.profile_get()
ctx.profile_enable(False)
T = (m + 127) // 128
ctas = {"chol_panel": B * T * (T - 1) // 2, "trtri": B * T * (T - 1) // 2, "lauum_grad": B * T * (T + 1) // 2}
out = {"m": m, "pairs": B, "evaluations": REPS, "kernel_ms_per_eval": {k: round(v[0] / REPS, 4) for k, v in prof.items() if v[1]},
       "launches_per_eval": {k: v[1] // REPS for k, v in prof.items() if v[1]},
       "ctas_per_eval": ctas,
       "us_per_skipped_cta": {k: prof[k][0] / REPS * 1e3 / n for k, n in ctas.items()}}
print(json.dumps(out))
