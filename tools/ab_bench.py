"""A/B of two builds of libgpbo.so on the headline benchmark, in one process tree on one GPU.

    python tools/ab_bench.py OUT_DIR [--base tools/ab/libgpbo_base.so] [--reps 3] [--steps 3] [bench.py options ...]

Runs `bench.py --dump-outputs` alternately with the base build (selected through GPBO_LIB) and the in-tree build,
`--reps` times each, then checks that every output array of every new run equals the base runs' bit for bit, and
compares `value` and the per-class kernel times.  Because `bench.py` credits m^3/3 per kernel class to every evaluated
pair, also to those whose Cholesky failed and which therefore skip most of the work, one more (untimed) run of the
same fit through the in-tree build counts the evaluations that came back not positive definite, and the kernel
efficiencies are restated over the positive definite evaluations only.  Writes OUT_DIR/ab.json and OUT_DIR/bench_*.json;
the output dumps go to a temporary directory.
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(lib, dump, extra):
    env = dict(os.environ)
    env.pop("GPBO_LIB", None)
    if lib:
        env["GPBO_LIB"] = lib
    cmd = [sys.executable, "bench.py", "--dump-outputs", dump] + extra
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    if p.returncode != 0 or not lines:
        raise RuntimeError(f"bench.py failed ({p.returncode}): {p.stderr[-2000:]}")
    return json.loads(lines[-1])


def same_outputs(a, b):
    names = sorted(f for f in os.listdir(a) if f.endswith(".npy"))
    if names != sorted(f for f in os.listdir(b) if f.endswith(".npy")):
        return False, ["different file sets"]
    bad = [n for n in names if not np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)),
                                                   equal_nan=True)]
    return not bad, bad


def count_not_pd(steps, modes, points, starts):
    """Evaluations per round of the benchmark's timed fit and how many of them were not positive definite."""
    sys.path.insert(0, ROOT)
    from gpbo_pkg import pkg

    T, Y, bl, st, gp_of = pkg.workload.fit_workload(modes, points, starts)
    ctx = pkg.default_context(0)
    failed = []

    class Counting:
        def upload_problem(self, t, y):
            ctx.upload_problem(t, y)

        def lml_grad_resident(self, theta, g):
            lml, grad, s = ctx.lml_grad_resident(theta, g)
            failed.append(int((s != 0).sum()))
            return lml, grad, s

    live = []
    pkg.sharding.fit_pairs(Counting(), T, Y, bl, st, gp_of, max_rounds=steps, stats=live)
    return live, failed


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--base", default=os.path.join(ROOT, "tools", "ab", "libgpbo_base.so"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=3)
    args, extra = ap.parse_known_args()
    extra = ["--steps", str(args.steps)] + extra
    os.makedirs(args.out, exist_ok=True)
    tmp = tempfile.mkdtemp(prefix="gpbo_ab_")
    runs = {"base": [], "new": []}
    for i in range(args.reps):
        for name, lib in (("base", os.path.abspath(args.base)), ("new", None)):
            dump = os.path.join(tmp, f"{name}_{i}")
            r = run_bench(lib, dump, extra)
            with open(os.path.join(args.out, f"bench_{name}_{i}.json"), "w") as f:
                json.dump(r, f)
            runs[name].append((r, dump))
            print(f"{name} {i}: value {r['value']:.3f}", flush=True)

    equal = {}
    for i, (_, dn) in enumerate(runs["new"]):
        for j, (_, db) in enumerate(runs["base"]):
            ok, bad = same_outputs(db, dn)
            equal[f"new_{i} vs base_{j}"] = True if ok else bad
    vals = {k: [r["value"] for r, _ in v] for k, v in runs.items()}
    kms = {k: {c: [r["roofline"]["kernel_ms"].get(c, 0.0) for r, _ in v] for c in runs["base"][0][0]["roofline"]["kernel_ms"]}
           for k, v in runs.items()}
    med = {k: statistics.median(v) for k, v in vals.items()}
    out = {
        "values": vals, "median": med, "ratio_new_over_base": med["new"] / med["base"],
        "kernel_ms": kms,
        "kernel_ms_change": {c: statistics.median(kms["new"][c]) / statistics.median(kms["base"][c]) - 1.0
                             for c in kms["base"] if statistics.median(kms["base"][c]) > 0},
        "outputs_bit_identical": equal,
        "all_outputs_bit_identical": all(v is True for v in equal.values()),
        "bench_args": extra + ["--dump-outputs", "<tmp>"],
    }

    cfg = runs["new"][0][0]["config"]
    fit = runs["new"][0][0]["fit"]
    points = int(re.search(r"n=(\d+)", cfg["workload"]).group(1))
    live, failed = count_not_pd(args.steps, fit["gps"], points, fit["starts_per_gp"])
    evals, pd = sum(live), sum(live) - sum(failed)
    out["evaluations"] = {"live_per_round": live, "not_pd_per_round": failed, "total": evals, "positive_definite": pd,
                          "matches_bench": live == cfg["live_pairs_per_round"]}
    # the bench's fractions credit m^3/3 per class to all `evals`; over the positive definite evaluations only:
    for name in ("base", "new"):
        fr = [r["roofline"] for r, _ in runs[name]]
        out[f"frac_{name}"] = {
            "whole_eval_frac_bench": [x["whole_eval_frac"] for x in fr],
            "whole_eval_frac_pd": [x["whole_eval_frac"] * pd / evals for x in fr],
            "class_frac_bench": [x["class_frac_algorithmic"] for x in fr],
            "class_frac_pd": [{k: v * pd / evals for k, v in x["class_frac_algorithmic"].items()} for x in fr],
        }
    with open(os.path.join(args.out, "ab.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("values", "median", "ratio_new_over_base", "kernel_ms_change",
                                          "all_outputs_bit_identical", "evaluations")}))


if __name__ == "__main__":
    main()
