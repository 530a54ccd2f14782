#!/usr/bin/env python
"""bench.py -- headline benchmark of the step2_fitgps hot path (contract: see the task prompt / DESIGN.md §6).

Primary workload (the north star's scaling target): synthetic r = 64 modes x n = 8192 time points x 32 starts, a
FIXED GLOBAL batch of 2048 (mode, start) pairs -- the multi-start L-BFGS-B fit of all 64 GPs.  A *step* is one
lock-step round of that fit: LML + gradient (blocked FP64 Cholesky, K^-1, gradient traces) of every pair whose
optimiser is still running, the optimisers advanced with the results.  `--steps K` rounds are timed (each start is
thereby bounded to K evaluations; W warm-up rounds on one wave of pairs come first), then the per-GP best start is
selected and the posterior moments of all 64 GPs (state / ddt estimates, ddt covariance, predictive std at
m' = n points) are computed -- timed separately and reported as `fits_per_s` beside the per-round numbers.

With N > 1 ranks (torchrun) the same global batch is sharded: every rank holds the replicated optimiser pool, the
live pairs are cut into N equal slices every round, results are all-gathered over NCCL (32 B per pair) -- STRONG
scaling; `value` = evaluations of all ranks / time of the slowest rank.  `value` is timed with CUDA events on the
library's stream with (t, y) resident in HBM; `e2e` is the same K rounds through the host-pointer calls timed by the
wall clock INCLUDING the upload of (t, y) and, every round, the pinned H2D of the trial points and the D2H of the
results.

`--impl reference` times the reference's own CPU path for the same evaluation
(GaussianProcessRegressor.log_marginal_likelihood(theta, eval_gradient=True) driven exactly as
codebase/gpkernels.py does, through the oracle port) on the host cores, one evaluation per step.

`--extras` adds the secondary measurements (other workloads, rooflines of the other kernel classes; several minutes).
`--dump-outputs DIR` writes what the fit and the posterior moments returned as DIR/<name>.npy (float64), so that two
builds can be compared output for output: the inputs are generated from fixed seeds.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

T_START = time.time()
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
DUMP_BYTES = 60_000_000             # --dump-outputs writes at most this much (float64 data)

R_MODES, N_POINTS, N_STARTS = 64, 8192, 32
METRIC, UNIT = "gp_lml_grad_evals_per_sec", "evals/s"
WORKLOAD = ("synthetic r={r} modes x n={m} points x {S} starts, fixed global batch of {B} (mode,start) pairs "
            "(north star scaling target; configs[3] shape at n=8192); step = one lock-step L-BFGS-B round = "
            "LML+gradient of every live pair")


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "500"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx = float(p[1])
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gp_oracle as orc

    return orc


def _cpu_gp(t, y):
    """The reference's CPU evaluation path (oracle port of GP_RBFW: scikit-learn regressor, alpha = 0)."""
    orc = _oracle()
    from threadpoolctl import threadpool_info, threadpool_limits

    # torchrun exports OMP_NUM_THREADS=1; the reference arm uses every host core the BLAS can take
    threadpool_limits(limits=os.cpu_count())
    b = np.array([(1e-5, 1e5), (1e-5, 1e2), (1e-16, 1e2)])
    gp = orc.OracleGP(tuple(b[0]), tuple(b[1]), tuple(b[2]), 0)
    gp.gpr.optimizer = None
    gp.fit(t, y)                # only stores the training data (no optimisation)
    cores = max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    return gp, cores


def run_reference(args):
    """Reference arm: the reference's CPU evaluation of the same quantity, one (mode, start) evaluation per step."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from gpbo_pkg import pkg

    r, m, S = args.modes, args.points, args.starts
    T, Y, theta, _ = pkg.workload.eval_workload(r, m, S)
    gp, cores = _cpu_gp(T[0], Y[0])
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        gp.lml_grad(theta[it % theta.shape[0]])
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    per = sum(times) / len(times)
    val = 1.0 / per
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(r=r, m=m, S=S, B=r * S),
                   "sample": f"one of the {r * S} (mode, start) LML+grad evaluations per step (a positive definite "
                             "theta; the GPU arm's batch also holds the ~20 % not-PD start points, which the CPU "
                             "path abandons after the failed Cholesky)"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"sklearn log_marginal_likelihood(theta, eval_gradient=True), m={m}, one pair per step"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--modes", type=int, default=R_MODES)
    ap.add_argument("--points", type=int, default=N_POINTS)
    ap.add_argument("--starts", type=int, default=N_STARTS)
    ap.add_argument("--m-est", type=int, default=0, help="estimation points of the moments phase (0: = points)")
    ap.add_argument("--budget-s", type=float, default=760.0,
                    help="secondary measurements (N = 1) are skipped once the process has run this long")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extras", action="store_true", help="also run the secondary measurements (N = 1)")
    ap.add_argument("--no-extras", dest="extras", action="store_false")
    ap.add_argument("--no-config4", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the timed fit and the posterior moments returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    sys.dont_write_bytecode = True      # the source tree may be read-only: no __pycache__ next to the project's modules
    if args.impl == "reference":
        return run_reference(args)

    import torch

    from gpbo_pkg import pkg

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    group = True if world > 1 else None

    r, m, S, K, W = args.modes, args.points, args.starts, args.steps, args.warmup
    T, Y, bl, starts, gp_of = pkg.workload.fit_workload(r, m, S)           # the same global batch on every rank
    B = starts.shape[0]
    ctx = pkg.default_context(local)
    lib_stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    # FP64 tensor-pipe peak (DMMA issue rate), measured live: MEASURED_PEAKS.json has no FP64 entry.  Best of five
    # ~60 ms runs after a warm-up run (the first launch on a cold GPU sees ramping clocks and reads ~2 % low).
    ctx.dmma_peak(100000)
    dmma_runs = [ctx.dmma_peak(100000)[0] for _ in range(5)]
    dmma_peak = max(dmma_runs)

    # ---- warm-up: W rounds of one wave of pairs (kernels loaded, workspace allocated, clocks up) -------------------
    ctx.upload_problem(T, Y)
    nwarm = max(1, min(B // world, ctx.wave_capacity(m), 148))
    pd_theta = pkg.workload.eval_workload(r, m, S)[2]
    for _ in range(max(W, 1)):
        ctx.lml_grad_resident(pd_theta[:nwarm], gp_of[:nwarm])

    # ---- timed: K lock-step rounds of the global fit ------------------------------------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = ctx.launch_count
    ctx.profile_enable(True)
    live = []
    barrier()
    w_e2e0 = time.perf_counter()
    ctx.upload_problem(T, Y)                       # e2e: the H2D of (t, y) is inside; the device-timed value starts after it
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(lib_stream)
    res = pkg.sharding.fit_pairs(ctx, T, Y, bl, starts, gp_of, group=group, max_rounds=K, stats=live)
    e1.record(lib_stream)
    barrier()
    wall_e2e = time.perf_counter() - w_e2e0
    prof = ctx.profile_get()
    ctx.profile_enable(False)
    launches = ctx.launch_count - launches0
    clocks = sampler.stop()
    ms = max_over_ranks(e0.elapsed_time(e1))
    wall_e2e = max_over_ranks(wall_e2e)
    rounds = len(live)
    evals = int(sum(live))
    ms_per_step = ms / max(rounds, 1)
    value = evals / (ms * 1e-3)
    e2e = evals / wall_e2e

    # ---- per-GP selection + posterior moments of all GPs (timed separately; fits/s) ---------------------------------
    funs = np.where(np.isfinite(res["fun"]), res["fun"], np.inf).reshape(r, S)
    theta_sel = res["theta"].reshape(r, S, 3)[np.arange(r), funs.argmin(1)]
    n_est = args.m_est or m
    t_est = np.linspace(0.0, 1.0, n_est)
    barrier()
    w0 = time.perf_counter()
    mom = pkg.sharding.moments(ctx, T, Y, theta_sel, t_est, group=group, want_cov=True, keep_cov=False)
    own = pkg.sharding.shard_indices(r, rank, world)
    pred = None
    if own.size:
        pred = ctx.predict(T[own], Y[own], theta_sel[own], t_est)        # predictive mean / std (gpkernels.py:350-365)
    barrier()
    t_mom = max_over_ranks(time.perf_counter() - w0)
    fits_per_s = r / (wall_e2e + t_mom)

    # ---- roofline of the dominant kernel class (DESIGN.md §4) -------------------------------------------------------
    T_blocks = (m + 127) // 128
    m_pad = T_blocks * 128
    blk = 2.0 * 128 ** 3
    SYM, TRI_A, TRI_B = 136.0 / 256.0, 36.0 / 64.0, 40.0 / 64.0
    issued_pp = {
        "chol_diag": blk * SYM * sum(j for j in range(T_blocks)),
        "chol_panel": blk * sum((T_blocks - 1 - j) * (j + TRI_B) for j in range(T_blocks)),
        "trtri": blk * sum((i - j - 1) + TRI_B + TRI_A for i in range(1, T_blocks) for j in range(i)),
        "lauum_grad": blk * sum(i * ((T_blocks - i - 1) + TRI_A) + SYM * (T_blocks - i) for i in range(T_blocks)),
    }
    local_evals = int(res.get("local_evals", evals))
    dom = max(("chol_panel", "trtri", "lauum_grad"), key=lambda k: prof[k][0])
    flops_third = float(m_pad) ** 3 / 3.0
    launches_dom = max(prof[dom][1], 1)
    total_flops_dom = flops_third * local_evals        # all launches of that class over the timed region, this rank
    dom_ms = prof[dom][0] + (prof["chol_diag"][0] if dom == "chol_panel" else 0.0)      # potrf = diag + panel
    achieved = total_flops_dom / (max(dom_ms, 1e-9) * 1e-3) / 1e12
    traffic = traffic_launch = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        traffic, traffic_launch = tj.get(dom), tj.get("_launch", {}).get(dom)
    except Exception:
        pass
    kernel_total_ms = sum(v[0] for v in prof.values())
    roofline = {
        "bound": "tensor", "kernel": dom, "achieved": achieved, "peak": dmma_peak, "unit": "TFLOP/s",
        "frac": achieved / dmma_peak, "traffic": traffic, "traffic_launch": traffic_launch,
        "peak_source": "FP64 DMMA issue-rate micro-benchmark run in this process (gpbo_bench_dmma_peak); "
                       "MEASURED_PEAKS.json holds no FP64 figure; cuBLAS DGEMM rate beside it in dgemm_cublas_tflops",
        "peak_runs": [round(x, 3) for x in dmma_runs],
        "peak_arithmetic": 128e-12 * torch.cuda.get_device_properties(dev).multi_processor_count
                           * (clocks.get("sm_max_mhz") or 0.0) * 1e6,
        "flops_per_launch": total_flops_dom / launches_dom, "avg_launch_ms": dom_ms / launches_dom,
        "share_of_step": prof[dom][0] / max(kernel_total_ms, 1e-9),
        "whole_eval_tflops": evals * float(m) ** 3 / (ms * 1e-3) / 1e12,
        "whole_eval_frac": evals * float(m) ** 3 / (ms * 1e-3) / 1e12 / (dmma_peak * world),
        "kernel_time_share_of_wall": kernel_total_ms / max(e0.elapsed_time(e1), 1e-9),
        "dmma_issued_tflops": {k: issued_pp[k] * local_evals / (prof[k][0] * 1e-3) / 1e12
                               for k in issued_pp if prof[k][0] > 0},
        "class_frac_algorithmic": {
            "potrf": flops_third * local_evals / (max(prof["chol_diag"][0] + prof["chol_panel"][0], 1e-9) * 1e-3) / 1e12 / dmma_peak,
            "trtri": flops_third * local_evals / (max(prof["trtri"][0], 1e-9) * 1e-3) / 1e12 / dmma_peak,
            "lauum_grad": flops_third * local_evals / (max(prof["lauum_grad"][0], 1e-9) * 1e-3) / 1e12 / dmma_peak},
        "kernel_ms": {k: round(v[0], 3) for k, v in prof.items() if v[1]},
        "rank": rank,
    }

    h2d_round = 28.0 * evals / max(rounds, 1) / world       # theta (24 B) + gp_of (4 B) per live pair, per rank
    d2h_round = 36.0 * evals / max(rounds, 1) / world       # lml (8) + grad (24) + status (4)
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": rounds, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": WORKLOAD.format(r=r, m=m, S=S, B=B), "global_pairs": B,
                   "live_pairs_per_round": live, "evaluations": evals,
                   "sharding": "replicated optimiser pool; live pairs re-cut into N equal slices every round; "
                               "all-gather of [lml, grad] (32 B / pair) over NCCL" if world > 1 else "single GPU",
                   "l2": "inputs larger than L2 (each pair's 512 MiB factor streams from HBM)",
                   "staging": "TMA (cp.async.bulk.tensor)" if not os.environ.get("GPBO_NO_TMA") else "LDGSTS (GPBO_NO_TMA)",
                   "waves_per_round_per_rank": -(-(-(-max(live) // world)) // max(ctx.wave_capacity(m), 1)) if live else 0,
                   "warmup_rounds": f"{max(W, 1)} rounds of {nwarm} pairs (one wave) before the timed region"},
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d_round), "d2h_bytes_per_step": int(d2h_round),
                "h2d_bytes_once": int(T.nbytes + Y.nbytes), "seconds": wall_e2e,
                "note": "same K rounds by wall clock, including the upload of (t, y) and the per-round pinned H2D / D2H"},
        "fits_per_s": fits_per_s,
        "fit": {"gps": r, "starts_per_gp": S, "rounds": rounds, "seconds_rounds": wall_e2e, "seconds_moments": t_mom,
                "m_est": n_est, "bounded": f"each start bounded to {K} evaluations (--steps); posterior moments "
                                           "(state, ddt, ddt covariance, predictive mean/std) of all GPs included, sqrtW excluded (SURVEY 8d)",
                "best_lml_first4": (-funs.min(1))[:4].tolist(),
                "running_after_K": int((res["status"] == -1).sum()), "not_pd_at_start": int((res["status"] == 5).sum()),
                "moments_status_ok": int((mom["status"] == 0).sum())},
        "roofline": roofline,
    }

    if rank == 0 and args.dump_outputs:
        # every rank holds the same fit result and moments; the predictions are those of the GPs this rank owns.
        # Per pair, fun is inf where K was not positive definite at the start (status 5), so the objective is
        # written as the per-GP selection the moments use: the best LML and its theta.
        arrays = {f"fit_{k}": res[k] for k in ("theta", "status", "nfev", "nit")}
        arrays.update(fit_best_lml=-funs.min(1), fit_best_theta=theta_sel)
        arrays.update({f"moments_{k}": mom[k] for k in ("alpha", "state", "ddt", "status")})
        if pred is not None:
            arrays.update(predict_mean=pred[0], predict_std=pred[1], predict_gps=own)
        dump_outputs(args.dump_outputs, arrays)

    def have_time(need_s=0.0):
        return (time.time() - T_START) + need_s < args.budget_s

    if world > 1 and not args.no_config4:
        out["config4_sample"] = config4_sample(pkg, ctx, dist, rank, world, dev, dmma_peak, barrier, max_over_ranks)
    # cpu_baseline comes first (N = 1 only), then, with --extras, the secondary measurements, each only when its
    # estimated duration still fits --budget-s
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(pkg, T, Y, m, evals=2 if have_time(60.0) else 1)
    elif rank == 0:
        out["cpu_baseline"] = None
    if rank == 0 and world == 1 and args.extras:
        extras = (("evals_configs3", 25.0, lambda: evals_configs3(pkg, ctx, dev, dmma_peak)),
                  ("roofline_prediction", 15.0, lambda: prediction_roofline(pkg, ctx, dmma_peak)),
                  ("posterior_grid", 5.0, lambda: posterior_grid_sample(ctx)),
                  ("roofline_assembly", 15.0, lambda: assembly_roofline(ctx, dev)),
                  ("dgemm_cublas_tflops", 3.0, lambda: dgemm_rate(dev)),
                  ("fit_reference_configs", 10.0, lambda: fit_reference_configs(ctx)),
                  ("fit_sample", 30.0, lambda: fit_sample(pkg, ctx)))
        for name, need_s, fn in extras:
            if not have_time(need_s):
                out[name] = "skipped: time budget"
                continue
            try:
                out[name] = fn()
            except Exception as exc:  # a secondary measurement must never lose the headline line
                out[name] = f"failed: {type(exc).__name__}: {exc}"
    out["seconds_total"] = time.time() - T_START
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(path, arrays):
    """Each array as path/<name>.npy in float64; one larger than its share of DUMP_BYTES is replaced by a fixed,
    seeded sample of its flattened elements (the same positions for the same shape)."""
    os.makedirs(path, exist_ok=True)
    cap = DUMP_BYTES // (8 * len(arrays))
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def dgemm_rate(dev, n=8192):
    """cuBLAS DGEMM n^3 through torch.matmul: the library's achievable FP64 rate, beside the DMMA issue peak."""
    import torch

    a = torch.randn((n, n), dtype=torch.float64, device=dev)
    b = torch.randn((n, n), dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(3):
        torch.matmul(a, b)
    e1.record()
    torch.cuda.synchronize(dev)
    return 3 * 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12


def evals_configs3(pkg, ctx, dev, dmma_peak, r=64, m=4096, S=32, steps=2):
    """BASELINE configs[3] on one B200 (last round's headline, kept as a secondary key): LML + gradient of all
    64 x 32 pairs at fixed theta, device-resident, CUDA events on the launching stream."""
    import torch

    T, Y, theta, gp_of = pkg.workload.eval_workload(r, m, S)
    B = theta.shape[0]
    Td, Yd, thd = (torch.as_tensor(x, device=dev) for x in (T, Y, theta))
    gpd = torch.as_tensor(gp_of, device=dev)
    lml_d = torch.empty(B, dtype=torch.float64, device=dev)
    grad_d = torch.empty((B, 3), dtype=torch.float64, device=dev)
    st_d = torch.empty(B, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)

    def step():
        ctx.lml_grad_device(Td.data_ptr(), Yd.data_ptr(), r, m, thd.data_ptr(), gpd.data_ptr(), B, lml_d.data_ptr(),
                            grad_d.data_ptr(), st_d.data_ptr(), stream.cuda_stream)

    step()
    ctx.profile_enable(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    prof = ctx.profile_get()
    ctx.profile_enable(False)
    ms = e0.elapsed_time(e1) / steps
    third = float(m) ** 3 / 3.0 * B * steps
    cls = {"potrf": prof["chol_diag"][0] + prof["chol_panel"][0], "trtri": prof["trtri"][0],
           "lauum_grad": prof["lauum_grad"][0]}
    return {"workload": f"r={r} x n={m} x {S} starts, fixed theta, one step = all {B} pairs", "evals_per_s": B / (ms * 1e-3),
            "ms_per_step": ms, "whole_eval_frac": B * float(m) ** 3 / (ms * 1e-3) / 1e12 / dmma_peak,
            "class_frac_algorithmic": {k: third / (v * 1e-3) / 1e12 / dmma_peak for k, v in cls.items() if v > 0},
            "kernel_ms_per_step": {k: round(v[0] / steps, 3) for k, v in prof.items() if v[1]},
            "status_ok_pairs": int((st_d == 0).sum().item())}


def config4_sample(pkg, ctx, dist, rank, world, dev, dmma_peak, barrier, max_over_ranks, r=8, m=16384, S=32, K=4):
    """BASELINE configs[4]'s shape (n = 16384, 32 starts) with the mode count reduced from 256 to 8 so that it fits
    the bench's time budget: K lock-step rounds of the sharded fit (same code path as the primary workload)."""
    import torch

    T, Y, bl, starts, gp_of = pkg.workload.fit_workload(r, m, S, seed=4)
    live = []
    ctx.upload_problem(T, Y)
    th = pkg.workload.eval_workload(r, m, S, seed=4)[2]
    ctx.lml_grad_resident(th[:4], gp_of[:4])                      # allocation / warm-up
    lib_stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(lib_stream)
    pkg.sharding.fit_pairs(ctx, T, Y, bl, starts, gp_of, group=True, max_rounds=K, stats=live)
    e1.record(lib_stream)
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    evals = int(sum(live))
    return {"workload": f"configs[4] shape: n={m} x {S} starts, modes reduced 256 -> {r} (stated), {K} rounds, "
                        f"{r * S} pairs sharded over {world} GPUs", "evals_per_s": evals / (ms * 1e-3),
            "seconds": ms * 1e-3, "live_pairs_per_round": live,
            "whole_eval_frac": evals * float(m) ** 3 / (ms * 1e-3) / 1e12 / (dmma_peak * world)}


def fit_sample(pkg, ctx, r=4, m=4096, S=32):
    """Measured GP fits/s to CONVERGENCE on a bounded sub-workload: r modes x S starts, full L-BFGS-B + posterior
    moments (state, ddt, covariance, predictive mean/std; sqrtW excluded per SURVEY 8d)."""
    T, Y, bl, starts, gp_of = pkg.workload.fit_workload(r, m, S, seed=123)
    t0 = time.perf_counter()
    res = ctx.fit(T, Y, bl, starts, gp_of)
    t_fit = time.perf_counter() - t0
    funs = np.where(np.isfinite(res["fun"]), res["fun"], np.inf).reshape(r, S)
    best = res["theta"].reshape(r, S, 3)[np.arange(r), funs.argmin(1)]
    t1 = time.perf_counter()
    ctx.lstsq_moments(T, Y, best, np.linspace(0, 1, m))
    ctx.predict(T, Y, best, np.linspace(0, 1, m))
    t_mom = time.perf_counter() - t1
    return {"modes": r, "starts": S, "m": m, "m_est": m, "fit_seconds": t_fit, "moments_seconds": t_mom,
            "fits_per_s": r / (t_fit + t_mom), "lml_grad_evals": res["evals"], "rounds": res["rounds"],
            "evals_per_s_over_fit": res["evals"] / t_fit, "best_lml": (-funs.min(1)).tolist()}


def assembly_roofline(ctx, dev):
    """HBM-write roofline of the stand-alone kernel-matrix assembly: 8 B per element, EVERY kind, the symmetric and the
    general kernel, at 8 x 8192^2, 2 x 16384^2 and the reference's own m' >> m shape (3200 x 200)."""
    import torch

    peaks = measured_peaks() or {}
    peak = float(peaks.get("hbm_gbs", 6543.1))
    stream = torch.cuda.current_stream(dev)
    names = {0: "K_train", 1: "K_yy", 2: "K_cross", 3: "kappa", 4: "K_zy", 5: "K_zz", 6: "dK_dlogell"}
    res = {}

    def run(kind, t1, t2, th, o, n1, n2, B, reps):
        # kernel time = the library's own CUDA events around each launch on the launching stream (gpbo_assemble
        # synchronises the stream before it returns, which an outer pair of events would count as kernel time)
        a = (kind, t1.data_ptr(), n1, n1, t2.data_ptr(), n2, n2, th.data_ptr(), B, o.data_ptr(), stream.cuda_stream)
        ctx.assemble_device(*a)
        ctx.assemble_device(*a)
        torch.cuda.synchronize(dev)
        ctx.profile_enable(True)
        for _ in range(reps):
            ctx.assemble_device(*a)
        ms, launches = ctx.profile_get()["assemble"]
        ctx.profile_enable(False)
        return launches * B * n1 * n2 * 8 / (ms * 1e-3) / 1e9

    def fill_rate(o, reps=10):
        # write-only streaming rate of the same buffer (cudaMemset through torch): context for the 8 B / element bound
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o.zero_()
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            o.zero_()
        e1.record()
        torch.cuda.synchronize(dev)
        return reps * o.numel() * 8 / (e0.elapsed_time(e1) * 1e-3) / 1e9

    fills = {}
    for label, B, n1, n2, reps in (("8x8192x8192", 8, 8192, 8192, 10), ("2x16384x16384", 2, 16384, 16384, 10),
                                   ("64x3200x200", 64, 3200, 200, 30)):
        t1 = torch.sort(torch.rand(B, n1, dtype=torch.float64, device=dev), dim=1).values.contiguous()
        t2 = t1.clone() if n1 == n2 else torch.sort(torch.rand(B, n2, dtype=torch.float64, device=dev), dim=1).values.contiguous()
        th = torch.log(torch.tensor([[1.5, 0.05, 1e-2]], dtype=torch.float64, device=dev)).repeat(B, 1).contiguous()
        o = torch.empty((B, n1, n2), dtype=torch.float64, device=dev)
        fills[label] = round(fill_rate(o) / peak, 4)
        for kind in range(7):
            if n1 != n2 and kind in (0, 1, 5, 6):
                continue                      # square-only kinds
            gen = run(kind, t1, t2, th, o, n1, n2, B, reps)
            res[f"{names[kind]}_general_{label}"] = round(gen / peak, 4)
            if n1 == n2:
                sym = run(kind, t1, t1, th, o, n1, n2, B, reps)
                res[f"{names[kind]}_symmetric_{label}"] = round(sym / peak, 4)
        del o
    fr = [v for v in res.values()]
    return {"bound": "hbm", "unit": "fraction of peak GB/s", "peak": peak, "bytes_per_element": 8,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy bandwidth)" if peaks else "fallback 6543.1 GB/s",
            "min_frac": min(fr), "min_frac_square": min(v for k, v in res.items() if "3200" not in k), "frac": res,
            "memset_frac": fills,
            "note": "frac = 8 B x elements / kernel time (library CUDA events, mean of 10-30 launches) / copy peak; "
                    "memset_frac = cudaMemset of the same buffer against the same peak (a write-only stream runs above "
                    "the read+write copy figure on these boxes)"}


def prediction_roofline(pkg, ctx, dmma_peak, G=8, m=4096):
    """compute_lstsq_matrices + predict for G GPs at m = m': per-class device time against the bound of each class --
    FP64 tensor peak for the Cholesky / prediction TRSM (m^2 m' flops) / Schur complement (m m'^2 flops), FP64 issue
    + HBM for the fused mean / std kernels, Newton-Schulz sqrtW as issued DMMA TFLOP/s."""
    T, Y, _, _ = pkg.workload.eval_workload(G, m, 1, seed=321)
    theta = np.tile(np.log([1.5, 0.05, 1e-2]), (G, 1))
    t_est = np.linspace(0, 1, m)
    ctx.lstsq_weights(T[:1], Y[:1], theta[:1], t_est, 1e-8)          # warm-up / allocation
    ctx.profile_enable(True)
    t0 = time.perf_counter()
    state, ddt, cov, w, st, wst, wit = ctx.lstsq_weights(T, Y, theta, t_est, 1e-8)
    dt = time.perf_counter() - t0
    prof = ctx.profile_get()
    ctx.profile_enable(False)
    ctx.profile_enable(True)
    ctx.predict(T, Y, theta, t_est)
    prof_p = ctx.profile_get()
    ctx.profile_enable(False)
    A = cov[0] + 1e-8 * np.eye(m)
    x = np.random.default_rng(0).standard_normal(m)
    resid = float(np.abs(w[0] @ (A @ (w[0] @ x)) - x).max() / np.abs(x).max())     # sqrtW (C + eta I) sqrtW x = x
    T_blocks = (m + 127) // 128
    ns_flops = float(wit.max() + 1) * G * 2.0 * 128 ** 3 * T_blocks * (T_blocks ** 2 + T_blocks * (T_blocks + 1))
    mp = T_blocks * 128
    hbm_peak = float((measured_peaks() or {}).get("hbm_gbs", 6543.1))
    tf = lambda flops, ms: flops / (ms * 1e-3) / 1e12 if ms > 0 else None
    trsm = tf(G * float(mp) ** 3, prof["cross_panel"][0])
    schur = tf(G * float(mp) ** 3, prof["schur"][0])
    return {"gps": G, "m": m, "m_est": m, "host_call_seconds": dt,
            "device_ms": {k: round(v[0], 3) for k, v in prof.items() if v[1]},
            "predict_device_ms": {k: round(v[0], 3) for k, v in prof_p.items() if v[1]},
            "trsm": {"bound": "tensor", "achieved": trsm, "peak": dmma_peak, "unit": "TFLOP/s",
                     "frac": trsm / dmma_peak if trsm else None, "flops": "m^2 m' per GP"},
            "schur": {"bound": "tensor", "achieved": schur, "peak": dmma_peak, "unit": "TFLOP/s",
                      "frac": schur / dmma_peak if schur else None, "flops": "m m'^2 per GP"},
            # fused means: kappa_zy alpha and K_zy alpha are generated on the fly, never stored -- FP64-issue bound; the
            # "materialised equivalent" is what reading the two m' x m matrices once from HBM would cost (the
            # reference's formulation, 16 m m' B per GP), i.e. the fused kernels run at this multiple of that roofline
            "mean": {"bound": "fp64 issue (exp per element; nothing read from HBM)", "ms": prof["mean_std"][0],
                     "elements_per_s": 2.0 * G * m * m / (prof["mean_std"][0] * 1e-3) if prof["mean_std"][0] > 0 else None,
                     "materialised_equivalent_gbs": 16.0 * G * m * m / (prof["mean_std"][0] * 1e-3) / 1e9
                     if prof["mean_std"][0] > 0 else None},
            # predictive std: row norms of V^T (m' x m per GP) read once from HBM
            "std": {"bound": "hbm", "ms": prof_p["std"][0], "unit": "GB/s", "peak": hbm_peak,
                    "achieved": 8.0 * G * mp * m / (prof_p["std"][0] * 1e-3) / 1e9 if prof_p["std"][0] > 0 else None,
                    "frac": 8.0 * G * mp * m / (prof_p["std"][0] * 1e-3) / 1e9 / hbm_peak if prof_p["std"][0] > 0 else None},
            "mean_std_ms": prof["mean_std"][0],
            "sqrtw_iterations": int(wit.max()), "sqrtw_status_ok": int((wst == 0).sum()),
            "sqrtw_ms": prof["sqrtw"][0], "sqrtw_identity_residual": resid,
            "sqrtw_dmma_issued_tflops": tf(ns_flops, prof["sqrtw"][0])}


def posterior_grid_sample(ctx, d=45, nreg=81):
    """Step-3 posterior assembly (SURVEY 8f N3) for the 8 weight matrices left resident by prediction_roofline (m' = 4096):
    posterior means, precisions and their Cholesky factors of all operator rows for the reference's 81-point regularizer
    grid (PDEs/step3_estimate.py:22: logspace(-16, 4, 81)) in one call; operator rows of length d = 45 (r = 8 quadratic)."""
    G, n = 8, 4096
    rng = np.random.default_rng(5)
    regs = np.logspace(-16, 4, nreg)
    W, where = None, "resident in HBM from the preceding lstsq_weights call"
    D = rng.standard_normal((n, d))
    rhs = rng.standard_normal((G, n))
    try:
        ctx.posterior_grid(D, rhs, regs[:2])                 # warm-up / allocation
    except Exception:                                        # the stack was evicted by a later call: bring own weights
        n = 1024
        M = rng.standard_normal((G, n, n))
        W = np.einsum("gij,gkj->gik", M, M) / n + 0.1 * np.eye(n)
        D, rhs, where = D[:n], rhs[:, :n], "host array (H2D inside the call)"
        ctx.posterior_grid(D, rhs, regs[:2], sqrtW=W)
    t0 = time.perf_counter()
    res = ctx.posterior_grid(D, rhs, regs, sqrtW=W)
    dt = time.perf_counter() - t0
    return {"modes": G, "m_est": n, "row_length": d, "regularizers": nreg, "host_call_seconds": dt,
            "not_positive_definite": int(res["status"].sum()), "candidates_per_s": nreg / dt, "weights": where}


def fit_reference_configs(ctx):
    """Full step2 fit (all 101 starts per GP, the reference's own start points) + posterior moments on five of the
    reference's experiment configurations (tests/golden/*.npz), with the reference's CPU wall time recorded when the
    fixtures were generated (8-core build container) beside it."""
    out = {}
    for name in ("seird_090_090_10_360", "seird_120_010_05_480", "heat_1_20_05_80_5", "euler_006_200_03_400_6",
                 "euler_006_050_01_400_6"):
        g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"), allow_pickle=False)
        T, Y, t_est = g["T"], g["Y"], g["t_est"]
        G = T.shape[0]
        bl = np.log(g["bounds"])
        S = g["starts"].shape[1] + 1
        starts = np.zeros((G, S, 3))
        starts[:, 1:] = g["starts"]
        gp_of = np.repeat(np.arange(G, dtype=np.int32), S)
        best_dt, res = None, None
        for _ in range(2):                       # second run: kernels loaded, buffers allocated
            t0 = time.perf_counter()
            res = ctx.fit(T, Y, bl, starts.reshape(-1, 3), gp_of)
            funs = np.where(np.isfinite(res["fun"]), res["fun"], np.inf).reshape(G, S)
            best = res["theta"].reshape(G, S, 3)[np.arange(G), funs.argmin(1)]
            t1 = time.perf_counter()
            ctx.lstsq_moments(T, Y, best, t_est)
            ctx.predict(T, Y, best, t_est)
            dt = time.perf_counter() - t0
            fit_dt = t1 - t0
            best_dt = dt if best_dt is None else min(best_dt, dt)
        lml = -funs.min(1)
        out[name] = {"gps": int(G), "m": int(T.shape[1]), "m_est": int(t_est.size), "starts": int(S),
                     "seconds": best_dt, "fit_seconds": fit_dt, "fits_per_s": G / best_dt,
                     "lml_grad_evals": res["evals"], "longest_chain": res["rounds"],
                     "max_rel_lml_gap_vs_reference": float(np.max((g["lml_opt"] - lml) / np.abs(g["lml_opt"]))),
                     "reference_cpu_fit_seconds": float(np.sum(g["fit_seconds"]))}
    return out


def cpu_baseline(pkg, T, Y, m, evals=2):
    """Oracle port (sklearn-driven, as the reference) timed on this box's host cores, bounded sample."""
    theta = pkg.workload.eval_workload(2, m, 2)[2]
    gp, cores = _cpu_gp(T[0], Y[0])
    times = []
    for k in range(evals):
        t0 = time.perf_counter()
        gp.lml_grad(theta[k])
        times.append(time.perf_counter() - t0)
    per = min(times)
    return {"value": 1.0 / per, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{evals} single-pair LML+grad evaluation(s) at m={m} via sklearn "
                      "GaussianProcessRegressor.log_marginal_likelihood (the fastest)",
            "host_cpus": os.cpu_count()}


if __name__ == "__main__":
    main()
