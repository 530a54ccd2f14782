"""Every way into the LML evaluation gives the same bits, and closing a context gives all its device memory back."""
import numpy as np
import pytest

import gp_oracle as orc

B = 12
FAIL = 5                                  # pair (and GP) whose kernel matrix is not positive definite
TH_FAIL = np.log([1.0, 0.1, 1e-17])       # sigma^2 = 1, ell = 0.1, chi below half an ulp of 1
GOOD_LO, GOOD_HI = np.log([0.3, 0.01, 1e-2]), np.log([3.0, 0.1, 1e-1])


def _batch(m):
    """B GPs, pair b on GP b.  GP FAIL has abscissae 10 apart (every off-diagonal kernel value underflows to 0 at
    ell = 0.1) with one repeated, so with TH_FAIL its pivot there is exactly 1 - 1 * 1 = 0."""
    t, y = orc.synthetic_trajectories(B, m, seed=m)
    T = np.tile(t, (B, 1))
    T[FAIL] = 10.0 * np.arange(m)
    T[FAIL, m // 2] = T[FAIL, m // 2 - 1]
    theta = np.random.default_rng(m).uniform(GOOD_LO, GOOD_HI, size=(B, 3))
    theta[FAIL] = TH_FAIL
    return T, y, theta


@pytest.mark.gpu
@pytest.mark.parametrize("m", [90, 1000])
def test_entry_points_agree_bitwise(ctx, m):
    """lml_grad (with and without gp_of), upload_problem + lml_grad_resident and lml_grad_device on torch tensors.  At
    m = 1000 the workspace holds only a few pairs, so the batch runs in several waves."""
    import torch
    from gpbo_pkg import pkg

    T, y, theta = _batch(m)
    gp = np.arange(B, dtype=np.int32)
    runs = {True: [], False: []}          # with_grad -> [(lml, grad, status)]
    c = pkg.Context(0, max_workspace_bytes=48 << 20)
    try:
        c.set_small_path(ctx.small_max)
        if m > 224:
            assert 1 < c.wave_capacity(m) < B
        for with_grad in (True, False):
            for g in (None, gp):
                runs[with_grad].append(c.lml_grad(T, y, theta, g, with_grad=with_grad))
        c.upload_problem(T, y)
        runs[True].append(c.lml_grad_resident(theta, gp))
        dev = torch.device("cuda", 0)
        Td, yd, thd, gpd = (torch.as_tensor(a, device=dev) for a in (T, y, theta, gp))
        stream = torch.cuda.current_stream(dev)
        for with_grad in (True, False):
            for g in (None, gpd):
                lml = torch.empty(B, dtype=torch.float64, device=dev)
                grad = torch.empty((B, 3), dtype=torch.float64, device=dev)
                st = torch.empty(B, dtype=torch.int32, device=dev)
                c.lml_grad_device(Td.data_ptr(), yd.data_ptr(), B, m, thd.data_ptr(), None if g is None else g.data_ptr(),
                                  B, lml.data_ptr(), grad.data_ptr() if with_grad else None, st.data_ptr(),
                                  stream.cuda_stream)
                runs[with_grad].append((lml.cpu().numpy(), grad.cpu().numpy() if with_grad else None, st.cpu().numpy()))
    finally:
        c.close()
    for with_grad, got in runs.items():
        lml0, grad0, st0 = got[0]
        assert st0[FAIL] != 0 and np.all(np.delete(st0, FAIL) == 0) and np.all(np.isfinite(np.delete(lml0, FAIL)))
        for k, (lml, grad, st) in enumerate(got[1:], 1):
            assert np.array_equal(st, st0) and np.array_equal(lml, lml0), (with_grad, k)
            if with_grad:
                assert np.array_equal(grad, grad0), k


@pytest.mark.gpu
def test_close_frees_device_memory():
    """Three contexts in turn run a fit on each path, a prediction, the step-2 weights and the step-3 posterior grid,
    and are closed.  The device's free memory must come back each time (the first round also loads the kernels)."""
    import torch
    from gpbo_pkg import pkg

    G, m, S = 2, 1000, 4
    t, y = orc.synthetic_trajectories(G, m, seed=4)
    T = np.tile(t, (G, 1))
    bl = np.log(np.array([(1e-5, 1e5), (1e-5, 1e2), (1e-16, 1e2)]))
    starts = np.random.default_rng(4).uniform(GOOD_LO, GOOD_HI, size=(G * S, 3))
    gp_of = np.repeat(np.arange(G, dtype=np.int32), S)
    opts = np.array([1e7, 1e-5, 15, 30, 20])
    t_est = np.linspace(0.0, 1.0, 300)

    def round_trip():
        c = pkg.Context(0)
        try:
            res = c.fit(T, y, bl, starts, gp_of, opts)                       # blocked path
            c.fit(T[:, :90], y[:, :90], bl, starts, gp_of, opts)             # in-shared small path
            theta = res["theta"][::S]
            c.predict(T, y, theta, t_est)
            state, ddt, _, w, _, wst, _ = c.lstsq_weights(T, y, theta, t_est, 1e-8)
            assert not wst.any()
            D = np.stack([np.ones_like(state[0]), state[0], state[0] ** 2], axis=1)
            c.posterior_grid(D, ddt, [1e-2, 1.0])                          # weights resident in HBM
        finally:
            c.close()
        torch.cuda.synchronize()
        return torch.cuda.mem_get_info(0)[0]

    round_trip()
    start = torch.cuda.mem_get_info(0)[0]
    for _ in range(3):
        assert abs(round_trip() - start) <= 8 << 20
