"""The batch-, size- and workspace-dependent schedules of the blocked path against the oracle.

The blocked path picks its schedule per launch from the batch size, the matrix size, the workspace limit and the SM
count (gpbo_api.cu): split-K plans (`plan_split`: unsplit, "fill the SMs" or quantisation-aware), the inverse rows on
the side stream (`eval_wave`), the wave sizes (`wave_capacity`) and the prediction TRSM (`moments_device`: one
persistent `cross_sweep_kernel`, or per-column launches with split-K mode 2).  A wrong chunk bound, a skipped partial
or an off-by-one in `sweep_locate` changes results only at the batch sizes that select that path.

This file restates the host schedule in Python (pinned by a CPU test to the worked numbers of the code comments and
DESIGN.md), derives every GPU case from the device's SM count, proves through the per-class launch counts that the
intended schedule ran, and compares the results with the CPU oracle at the suite's usual bars.
"""
import contextlib
import functools

import numpy as np
import pytest

import gp_oracle as orc
from conftest import record

# ---- Python restatement of the host schedule (gpbo_api.cu) ---------------------------------------------------------
TB, BK = 128, 16                      # tile edge, k-slice (common.cuh)
SLICES = TB // BK                     # k-slices per block column
SPLIT_MAX, SPLIT_MIN = 16, 4          # plan_split: most chunks, fewest slices per chunk
QUANT_MAX, QUANT_COST, QUANT_GAIN = 8, 0.02, 0.97   # quantisation-aware branch: most chunks, cost per chunk, gain
PAIR_PARAMS_BYTES = 40                # sizeof(PairParams)
MIB = 1 << 20


def _cdiv(a, b):
    return -(-a // b)


def pad(m):
    return _cdiv(m, TB) * TB


def sm_fill_split(units, nk_max, sms):
    """Chunks of plan_split's "fill the SMs" rule (before the quantisation-aware branch)."""
    return min(SPLIT_MAX, sms // units, nk_max // SPLIT_MIN)


def plan_split(units, nk_max, sms):
    """Chunks per tile of one launch of `units` tiles with a k-loop of nk_max slices; 1: no partial launch."""
    if units <= 0 or nk_max < 16:
        return 1
    nsplit = sm_fill_split(units, nk_max, sms)
    if nsplit < 2 and units <= 4 * sms:
        best, nsplit = float(_cdiv(units, sms)), 1
        ns = 2
        while ns <= QUANT_MAX and nk_max // ns >= 2 * SPLIT_MIN:
            cost = float(_cdiv(units * ns, sms)) / ns + QUANT_COST * ns
            if cost < QUANT_GAIN * best:
                best, nsplit = cost, ns
            ns += 1
    if nsplit < 2:
        return 1
    chunk = _cdiv(nk_max, nsplit)
    return _cdiv(nk_max, chunk)


def split_branch(units, nk_max, sms):
    """None (no split), "sms" (fill the SMs) or "quantised": which branch of plan_split chose the launch's plan."""
    if plan_split(units, nk_max, sms) < 2:
        return None
    return "sms" if sm_fill_split(units, nk_max, sms) >= 2 else "quantised"


def pair_bytes(m_pad):
    T = m_pad // TB
    ntiles = T * (T + 1) // 2
    return m_pad * m_pad * 8 + 2 * T * TB * TB * 8 + 3 * m_pad * 8 + T * 8 + ntiles * 32 + PAIR_PARAMS_BYTES + 16


def wave_sizes(want, limit, m_pad, extra, reserved, sms):
    """Pairs of each wave (wave_capacity + the callers' loops); [] when one pair does not fit."""
    per = pair_bytes(m_pad) + extra
    if limit <= reserved + per:
        return []
    cap = (limit - reserved) // per
    if cap < want:
        nw = _cdiv(want, cap)
        cap = _cdiv(want, nw)
        up = _cdiv(cap, sms) * sms
        if up <= (limit - reserved) // per:
            cap = up
    return [min(cap, want - w0) for w0 in range(0, want, cap)]


def lml_reserved(G, m):
    """Workspace lml_grad_device keeps outside the waves: the padded targets of G GPs and 1 MiB."""
    return G * pad(m) * 8 + MIB


def moments_extra_reserved(G, m, n, predict, cov):
    """(per-pair extra, reserved) of moments_device: X (prediction, or a covariance) and the scaled evaluation points
    per GP; the covariance staging of all G GPs beside the waves."""
    m_pad, n_pad = pad(m), pad(n)
    extra = (n_pad * m_pad * 8 if predict or cov else 0) + n_pad * 8
    return extra, G * m_pad * 8 + MIB + (G * n * n * 8 if cov else 0)


def overlap(nb, m, sms, with_grad=True):
    """Whether eval_wave runs the inverse rows (and their split-K partials) on the side stream."""
    return with_grad and nb <= sms and pad(m) // TB >= 4


def sweep_taken(nb, n, sms):
    return 2 * nb * (pad(n) // TB) >= sms


def column_plans(m, nb, sms):
    """[(nk_max, nsplit, branch)] of factorisation columns j = 0 .. T-1 (mode 0)."""
    T = pad(m) // TB
    return [(SLICES * j, plan_split(nb * (T - j), SLICES * j, sms), split_branch(nb * (T - j), SLICES * j, sms))
            for j in range(T)]


def row_plans(m, nb, sms):
    """[(nk_max, nsplit, branch)] of inverse rows i = 1 .. T-1 (mode 1)."""
    T = pad(m) // TB
    return [(SLICES * i, plan_split(nb * i, SLICES * i, sms), split_branch(nb * i, SLICES * i, sms))
            for i in range(1, T)]


def cross_plans(m, nb, n, sms):
    """[(nk_max, nsplit, branch)] of the per-column prediction TRSM (mode 2)."""
    T, xT = pad(m) // TB, pad(n) // TB
    return [(SLICES * j, plan_split(nb * xT, SLICES * j, sms), split_branch(nb * xT, SLICES * j, sms))
            for j in range(T)]


def expected_launches(m, waves, sms, with_grad=True, n=None):
    """Per-class launch counts of one call: lml_grad (n None) or a posterior-moment call with n evaluation points."""
    T = pad(m) // TB
    out = dict(chol_diag=0, chol_panel=0, trtri=0, cross_panel=0)
    for nb in waves:
        out["chol_diag"] += T
        out["chol_panel"] += T - 1 + sum(ns > 1 for _, ns, _ in column_plans(m, nb, sms))
        if n is None and with_grad:
            out["trtri"] += T - 1 + sum(ns > 1 for _, ns, _ in row_plans(m, nb, sms))
        if n is not None:
            if sweep_taken(nb, n, sms):
                out["cross_panel"] += 1
            else:
                out["cross_panel"] += T + sum(ns > 1 for _, ns, _ in cross_plans(m, nb, n, sms))
    return out


def sweep_locate(b, T):
    """(unit, step) where the cost offset b falls: the smallest step j with j (j + 1) >= the offset inside the unit."""
    C = T * (T + 1)
    u, rem = divmod(b, C)
    j = 0
    while j * (j + 1) < rem:
        j += 1
    if j >= T:
        u, j = u + 1, 0
    return u, j


def sweep_ranges(units, T, grid):
    """(u0, j0, u1, j1) of every CTA of cross_sweep_kernel: the range starts in unit u0 at step j0 and ends in u1
    before step j1."""
    W = units * T * (T + 1)
    return [sweep_locate(W * b // grid, T) + sweep_locate(W * (b + 1) // grid, T) for b in range(grid)]


def sweep_segments(units, T, grid):
    """Per CTA, the (unit, first step, end step) segments in execution order: head of u1, whole units, tail of u0."""
    out = []
    for u0, j0, u1, j1 in sweep_ranges(units, T, grid):
        split_tail, split_head = j0 > 0, j1 > 0 and u1 < units
        first_whole = u0 + 1 if split_tail else u0
        segs = [(u1, 0, j1)] if split_head else []
        segs += [(u, 0, T) for u in range(first_whole, u1)]
        segs += [(u0, j0, T)] if split_tail else []
        out.append(segs)
    return out


def sweep_labels(units, T, grid):
    """Which of the sweep's cuts occur: all-whole, no-whole-unit (a CTA with only a head and a tail), one-step-head,
    last-step-tail, T=1."""
    labels = set()
    if T == 1:
        labels.add("T=1")
    split = False
    for (u0, j0, u1, j1), segs in zip(sweep_ranges(units, T, grid), sweep_segments(units, T, grid)):
        if j0 > 0 or (j1 > 0 and u1 < units):
            split = True
        if not any(ja == 0 and jb == T for _, ja, jb in segs):
            labels.add("no-whole-unit")
        if j1 == 1 and u1 < units:
            labels.add("one-step-head")
        if 0 < j0 == T - 1:
            labels.add("last-step-tail")
    if not split:
        labels.add("all-whole")
    return labels


# ---- CPU: the model against the worked numbers ----------------------------------------------------------------------
def test_schedule_model_worked_numbers():
    # "256 tiles on 148 SMs take two tile times ... 4 chunks: 1.75" (plan_split)
    assert plan_split(256, 64, 148) == 4 and split_branch(256, 64, 148) == "quantised"
    assert plan_split(1, 56, 148) == 14 and split_branch(1, 56, 148) == "sms"
    assert plan_split(148, 56, 148) == 1 and plan_split(8, 8, 148) == 1      # one full round; k-loop too short
    # re-derived chunk count: 48 slices in 5 chunks of 10, the last one 8 long
    assert plan_split(80, 48, 148) == 5
    # "2048 pairs at a capacity of 1030 run as 1024 + 1024" (wave_capacity); at 1100 the SM rounding applies
    per = pair_bytes(4096)
    assert wave_sizes(2048, 1030 * per + MIB, 4096, 0, MIB, 148) == [1024, 1024]
    assert wave_sizes(2048, 1100 * per + MIB, 4096, 0, MIB, 148) == [1036, 1012]
    assert wave_sizes(5, 2 * per + MIB + per // 2, 4096, 0, MIB, 148) == [2, 2, 1]
    assert wave_sizes(1, per + MIB, 4096, 0, MIB, 148) == []
    # "256 units -> 148 CTAs" in sweep mode 0
    assert len(sweep_ranges(256, 2, min(256, 148))) == 148
    # the m = 1000 regimes of the GPU cases at 148 SMs
    assert not any(ns > 1 for _, ns, _ in column_plans(1000, 148, 148) + row_plans(1000, 148, 148))
    assert overlap(148, 1000, 148) and not overlap(149, 1000, 148)
    assert {b for _, _, b in column_plans(1000, 149, 148) + row_plans(1000, 149, 148)} == {None, "quantised"}
    ex, res = 0, lml_reserved(4, 1000)
    assert wave_sizes(400, res + 300 * pair_bytes(1024) + 1, 1024, ex, res, 148) == [296, 104]
    assert [ns for _, ns, _ in cross_plans(1000, 1, 73 * TB, 148)] == [1, 1, 2, 2, 2, 2, 2, 2]
    assert not sweep_taken(1, 73 * TB, 148) and sweep_taken(1, 74 * TB, 148)
    assert expected_launches(1000, [1], 148) == dict(chol_diag=8, chol_panel=13, trtri=13, cross_panel=0)


@pytest.mark.parametrize("units,T,grid", [(256, 2, 148), (150, 8, 148), (150, 1, 148), (102, 5, 102), (154, 5, 148),
                                          (84, 3, 84), (1000, 16, 148), (149, 32, 148)])
def test_sweep_segments_cover_every_step_once(units, T, grid):
    """The restated cut of the row sweep: every (unit, step) is computed exactly once, a unit is shared by at most two
    CTAs, and a tail's head is published by the CTA before it (which runs it first)."""
    done = np.zeros((units, T), dtype=int)
    owners = [set() for _ in range(units)]
    segs = sweep_segments(units, T, grid)
    for b, cta in enumerate(segs):
        assert cta, b
        for k, (u, ja, jb) in enumerate(cta):
            assert 0 <= ja < jb <= T
            done[u, ja:jb] += 1
            owners[u].add(b)
            if ja > 0:                                    # a tail: the previous CTA's first segment is its head
                assert k == len(cta) - 1 and segs[b - 1][0] == (u, 0, ja), (b, u)
    assert np.all(done == 1)
    assert max(len(o) for o in owners) <= 2


# ---- GPU cases ------------------------------------------------------------------------------------------------------
LIMIT = 8 << 30                       # one wave for every single-wave case below
NPD_THETA = np.log([1.0, 0.1, 1e-17])  # with abscissae 10 apart and one repeated: an exact zero pivot (not PD)
M1, M2 = 1000, 2048
# 4 GPs x 2 theta at m = 1000, 2 GPs x 1 theta at m = 2048; cond(K) <= 1e6 (asserted with the oracle)
THETA = {M1: np.log([[1.5, 0.05, 1e-2], [0.6, 0.1, 3e-2], [2.5, 0.03, 1e-2], [0.8, 0.2, 5e-2],
                     [1.2, 0.07, 2e-2], [3.0, 0.04, 3e-2], [0.5, 0.12, 1e-2], [1.8, 0.06, 4e-2]]),
         M2: np.log([[2.5, 0.05, 1e-2], [0.7, 0.03, 3e-2]])}


def rel(a, b, scale=None):
    a, b = np.asarray(a), np.asarray(b)
    s = np.abs(b).max() if scale is None else scale
    return np.abs(a - b).max() / max(s, 1e-300)


@functools.lru_cache(maxsize=None)
def _sms():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


@contextlib.contextmanager
def _context(limit, family=0):
    """A context of the test's own: blocked path for every size, launch counting on, closed at the end."""
    from gpbo_pkg import pkg

    c = pkg.Context(0, max_workspace_bytes=limit)
    try:
        c.set_small_path(0)
        c.set_kernel_family(family)
        c.profile_enable(True)
        yield c
    finally:
        c.close()


def _counts(c):
    return {k: n for k, (_, n) in c.profile_get().items()}


def _trajectories(G, m, seed):
    """G GPs with abscissae and targets of their own."""
    rows = [orc.synthetic_trajectories(1, m, seed=seed + g) for g in range(G)]
    return np.stack([t for t, _ in rows]), np.vstack([y for _, y in rows])


@functools.lru_cache(maxsize=None)
def _lml_problem(m):
    """(T, Y, theta, gp) of the distinct (GP, theta) pairs at size m: pair k uses GP gp[k]."""
    theta = THETA[m]
    G = 4 if m == M1 else 2
    T, Y = _trajectories(G, m, seed=10 * m)
    return T, Y, theta, np.arange(len(theta)) * G // len(theta)


def _kernel_matrix(family, t, theta):
    if family == 0:
        return orc.np_kernel(t, theta)
    s2, ell, chi = np.exp(theta)
    return orc.np_matern(t, t, s2, ell, family) + chi * np.eye(t.size)


@functools.lru_cache(maxsize=None)
def _lml_oracle(family, m, k):
    """Oracle LML and gradient of distinct pair k (computed once per module)."""
    T, Y, theta, gp = _lml_problem(m)
    t, y = T[gp[k]], Y[gp[k]]
    if family == 0:
        l0, g0, s0 = orc.np_lml_grad(t, y, theta[k])
    else:
        l0, g0, s0 = orc.np_lml_grad_matern(t, y, theta[k], family)
    ev = np.linalg.eigvalsh(_kernel_matrix(family, t, theta[k]))
    assert s0 == 0 and ev[-1] / ev[0] <= 1e6, (family, m, k, ev[-1] / ev[0])
    return l0, g0


def _lml_case(name, S):
    """m, pairs, kernel family, gradient, workspace limit, not-PD pair position and the regime check of a case."""
    case = dict(m=M1, nb=S // 4, family=0, with_grad=True, limit=LIMIT, notpd=None)
    if name == "sm_split_nb1":
        case.update(nb=1)
    elif name == "quantised_s8":
        case.update(nb=_cdiv(S, 8))
    elif name == "quantised_s4":
        pass
    elif name == "quantised_s2":
        case.update(nb=S // 2 + 1)
    elif name == "full_round":
        case.update(nb=S)
    elif name == "full_round_plus_one":
        case.update(nb=S + 1)
    elif name == "lml_only":
        case.update(with_grad=False)
    elif name == "matern32":
        case.update(family=3)
    elif name == "matern52_nb1":
        case.update(family=5, nb=1)
    elif name == "two_unequal_waves":
        cap = 2 * S + 4
        case.update(nb=2 * S + _cdiv(7 * S, 10), limit=lml_reserved(4, M1) + cap * pair_bytes(pad(M1)) + MIB)
    elif name == "notpd_in_quantised":
        case.update(notpd=S // 8)
    elif name == "m2048_mixed":
        case.update(m=M2, nb=8)
    else:
        raise ValueError(name)
    return case


def _check_lml_regime(name, case, waves, S):
    m, nb, wg = case["m"], case["nb"], case["with_grad"]
    plans = [(column_plans(m, w, S), row_plans(m, w, S) if wg else []) for w in waves]
    branches = [{b for _, _, b in cols} | {b for _, _, b in rows} for cols, rows in plans]
    if name == "two_unequal_waves":
        assert len(waves) == 2 and waves[0] % S == 0 and waves[0] > S >= waves[1], waves
        assert branches[0] == {None} and not overlap(waves[0], m, S)
        assert "quantised" in branches[1] and overlap(waves[1], m, S)
        return
    assert waves == [nb], waves
    cols, rows = plans[0]
    if name in ("sm_split_nb1", "matern52_nb1"):
        assert all(b == "sms" for nk, _, b in cols + rows if nk >= 16) and overlap(nb, m, S)
        # inverse rows: a chunk shorter than a block column puts a chunk boundary inside the DT block
        assert any(_cdiv(nk, ns) < SLICES for nk, ns, _ in rows if ns > 1)
    elif name in ("quantised_s8", "quantised_s4", "matern32", "notpd_in_quantised"):
        assert "quantised" in {b for _, _, b in cols} and "quantised" in {b for _, _, b in rows} and overlap(nb, m, S)
    elif name == "quantised_s2":
        assert branches[0] == {None, "quantised"} and overlap(nb, m, S)
    elif name == "full_round":
        assert branches[0] == {None} and overlap(nb, m, S)
    elif name == "full_round_plus_one":
        assert "quantised" in branches[0] and not overlap(nb, m, S)
    elif name == "lml_only":
        assert any(ns > 1 for _, ns, _ in cols) and not rows
    elif name == "m2048_mixed":
        assert branches[0] == {None, "sms", "quantised"} and overlap(nb, m, S)
        # shorter last chunks: the chunk count was re-derived from the rounded-up chunk length
        assert any(nk % _cdiv(nk, ns) for nk, ns, _ in cols + rows if ns > 1)


LML_CASES = ["sm_split_nb1", "quantised_s8", "quantised_s4", "quantised_s2", "full_round", "full_round_plus_one",
             "lml_only", "matern32", "matern52_nb1", "two_unequal_waves", "notpd_in_quantised", "m2048_mixed"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", LML_CASES)
def test_lml_grad_schedules_against_oracle(name):
    S = _sms()
    case = _lml_case(name, S)
    m, nb, family, wg = case["m"], case["nb"], case["family"], case["with_grad"]
    T, Y, theta, gp = _lml_problem(m)
    k = np.arange(nb) % len(theta)                 # distinct pair of every batch entry, repeated cyclically
    if family:                                     # the first theta of each GP (scikit-learn's Matern oracle is slow)
        k = k // 2 * 2
    th, gp_of = theta[k], gp[k].astype(np.int32)
    if case["notpd"] is not None:                  # one more GP: abscissae 10 apart with one repeated
        bad = 10.0 * np.arange(m)
        bad[m // 2] = bad[m // 2 - 1]
        T, Y = np.vstack([T, bad]), np.vstack([Y, Y[:1]])
        k[case["notpd"]] = -1
        th[case["notpd"]] = NPD_THETA
        gp_of[case["notpd"]] = T.shape[0] - 1
    G = T.shape[0]
    waves = wave_sizes(nb, case["limit"], pad(m), 0, lml_reserved(G, m), S)
    _check_lml_regime(name, case, waves, S)

    with _context(case["limit"], family) as c:
        lml, grad, st = c.lml_grad(T, Y, th, gp_of, with_grad=wg)
        counts = _counts(c)
    exp = expected_launches(m, waves, S, with_grad=wg)
    assert {key: counts[key] for key in exp} == exp, (name, S, waves)

    wave_size = np.repeat(waves, waves)            # copies in waves of one size ran the same split-K plans
    if case["notpd"] is not None:
        b = case["notpd"]
        assert st[b] == 1 and lml[b] == -np.inf and np.all(grad[b] == 0), (lml[b], grad[b], st[b])
    for kk in np.unique(k[k >= 0]):
        l0, g0 = _lml_oracle(family, m, int(kk))
        sel = np.flatnonzero(k == kk)
        assert np.all(st[sel] == 0), (name, kk)
        el = np.abs(lml[sel] - l0).max() / abs(l0)
        record(f"lml_rel[schedules, {name}]", el)
        assert el <= 1e-10, (name, kk, lml[sel], l0)
        if wg:
            eg = max(rel(g, g0, max(1.0, np.abs(g0).max())) for g in grad[sel])
            record(f"grad_rel[schedules, {name}]", eg)
            assert eg <= 1e-9, (name, kk, grad[sel], g0)
        for w in np.unique(wave_size[sel]):
            same = sel[wave_size[sel] == w]
            assert np.all(lml[same] == lml[same[0]]), (name, kk, w)
            if wg:
                assert np.all(grad[same] == grad[same[0]]), (name, kk, w)


# ---- posterior moments ----------------------------------------------------------------------------------------------
THETA_M = np.log([[2.5, 0.05, 1e-2], [0.7, 0.2, 3e-3], [1.3, 0.1, 5e-3], [0.9, 0.07, 4e-3]])


def _moment_case(name, S):
    """kind ("predict" / "lstsq"), family, m, G, per-GP points (G, n) or shared (n,), workspace limit."""
    half = _cdiv(S, 2)
    case = dict(kind="predict", family=0, limit=LIMIT)
    if name == "sweep_t1":                          # 150 units of one step each [S = 148]
        case.update(m=100, G=2, n=(S // 2 + 1) * TB - 100)
    elif name == "sweep_all_whole":                 # units <= S: one whole unit per CTA
        case.update(m=520, G=2, n=((S + 5) // 3) * TB - 28)
    elif name == "sweep_no_whole_unit":             # units just above S: head + tail, nothing whole in between
        case.update(m=1000, G=2, n=(S // 2 + 1) * TB - 100)
    elif name == "sweep_t2_many_units":
        case.update(m=200, G=8, n=(S * 7 // 32) * TB - 96)
    elif name == "per_column_below_threshold":
        case.update(m=1000, G=1, n=(half - 1) * TB)
    elif name == "sweep_at_threshold":
        case.update(m=1000, G=1, n=half * TB)
    elif name == "matern32_predict_sweep":
        case.update(family=3, m=520, G=2, n=(S // 2 + 3) * TB - 28)
    elif name == "matern52_lstsq_sweep":
        case.update(kind="lstsq", family=5, m=300, G=_cdiv(half, 12), n=1500)
    else:
        raise ValueError(name)
    case["t_est"] = np.linspace(-0.05, 1.05, case["n"])
    return case


def _moment_oracle(kind, family, t, y, theta, t_est):
    if kind == "predict":
        if family == 0:
            mean, std = orc.np_predict(t, y, theta, t_est)
            return dict(mean=mean, std=std, alpha=orc.np_alpha(t, y, theta)[0])
        mean, std, alpha = orc.np_predict_matern(t, y, theta, t_est, family)
        return dict(mean=mean, std=std, alpha=alpha)
    if family == 0:
        r = orc.np_lstsq_moments(t, y, theta, t_est, want_sqrtW=False)
    else:
        r = orc.np_lstsq_moments_matern(t, y, theta, t_est, family)
    return dict(state=r["state_estimate"], ddt=r["ddt_estimate"], cov=r["ddt_covariance"])


TOL_M = dict(mean=1e-10, std=1e-7, alpha=1e-9, state=1e-10, ddt=1e-10, cov=1e-9)


def _run_moments(kind, family, T, Y, theta, t_est, limit, S, tag):
    """One posterior-moment call on a context of its own: its waves and launch counts against the model, every GP
    against its own oracle.  Returns the waves."""
    G, m = T.shape
    n = t_est.shape[-1]
    extra, reserved = moments_extra_reserved(G, m, n, kind == "predict", kind == "lstsq")
    waves = wave_sizes(G, limit, pad(m), extra, reserved, S)
    with _context(limit, family) as c:
        if kind == "predict":
            mean, std, alpha, st = c.predict(T, Y, theta, t_est, want_alpha=True)
            got = dict(mean=mean, std=std, alpha=alpha)
        else:
            state, ddt, cov, st = c.lstsq_moments(T, Y, theta, t_est)
            got = dict(state=state, ddt=ddt, cov=cov)
        counts = _counts(c)
    exp = expected_launches(m, waves, S, n=n)
    assert {key: counts[key] for key in exp} == exp, (tag, S, waves)
    assert np.all(st == 0)
    for g in range(G):
        ref = _moment_oracle(kind, family, T[g], Y[g], theta[g], t_est if t_est.ndim == 1 else t_est[g])
        for key, r in ref.items():
            err = rel(got[key][g], r)
            record(f"{key}_rel[schedules, {tag}]", err)
            assert err <= TOL_M[key], (tag, g, key, err)
        if kind == "lstsq":
            assert np.array_equal(got["cov"][g], got["cov"][g].T)
    return waves


MOMENT_CASES = ["sweep_t1", "sweep_all_whole", "sweep_no_whole_unit", "sweep_t2_many_units",
                "per_column_below_threshold", "sweep_at_threshold", "matern32_predict_sweep", "matern52_lstsq_sweep"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", MOMENT_CASES)
def test_moments_schedules_against_oracle(name):
    S = _sms()
    case = _moment_case(name, S)
    m, G, n = case["m"], case["G"], case["n"]
    T_, xT, units = pad(m) // TB, pad(n) // TB, G * pad(n) // TB
    if name == "per_column_below_threshold":
        plans = cross_plans(m, G, n, S)
        assert not sweep_taken(G, n, S) and any(ns > 1 for _, ns, _ in plans), plans
    else:
        assert sweep_taken(G, n, S)
        labels = sweep_labels(units, T_, min(units, S))
        want = {"sweep_t1": {"T=1"}, "sweep_all_whole": {"all-whole"}, "sweep_no_whole_unit": {"no-whole-unit"},
                "sweep_t2_many_units": {"one-step-head", "last-step-tail"}}.get(name, set())
        assert want <= labels, (name, S, units, T_, labels)
        if name in ("sweep_t1", "sweep_t2_many_units"):
            assert units > S and T_ == (1 if name == "sweep_t1" else 2)
        if name == "matern32_predict_sweep":
            assert "all-whole" not in labels
    T, Y = _trajectories(G, m, seed=7 * m + xT)
    theta = THETA_M[np.arange(G) % len(THETA_M)]
    waves = _run_moments(case["kind"], case["family"], T, Y, theta, case["t_est"], case["limit"], S, name)
    assert waves == [G]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["predict", "lstsq"])
def test_moments_in_several_waves_with_per_gp_grids(kind):
    """G = 5 GPs under a workspace that holds 2: waves of 2 + 2 + 1, equispaced (Toeplitz K_zz) and jittered
    estimation grids mixed inside the waves; every GP against its own oracle, alpha and the covariance included."""
    S = _sms()
    G, m, n = 5, 300, 400
    rng = np.random.default_rng(5)
    grids = []
    for g in range(G):
        lo, hi = -0.02 * g, 1.0 + 0.01 * g
        grid = np.linspace(lo, hi, n)
        if g % 2:
            grid = np.sort(grid + 2e-4 * rng.standard_normal(n))
        grids.append(grid)
    t_est = np.stack(grids)
    extra, reserved = moments_extra_reserved(G, m, n, kind == "predict", kind == "lstsq")
    limit = reserved + 2 * (pair_bytes(pad(m)) + extra) + MIB
    assert wave_sizes(G, limit, pad(m), extra, reserved, S) == [2, 2, 1]
    T, Y = _trajectories(G, m, seed=77)
    theta = THETA_M[np.arange(G) % len(THETA_M)]
    assert _run_moments(kind, 0, T, Y, theta, t_est, limit, S, f"waves 2+2+1 {kind}") == [2, 2, 1]
