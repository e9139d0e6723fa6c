"""pmmh_flps_model_corr beyond the chain kernel: one problem with more than 4096 particles runs on the grid kernel
(csrc/sv_grid.cu) instantiated for the model (diag[PMMH_DIAG_KERNEL] == 5).

- Linear Gaussian bootstrap filter against the NumPy restatement (oracle/generic_pf.py) from N = 4097 to 2^16, for
  phi > 0, phi < 0 and phi = 0 (golden_inputs.LG_PARAM_SETS by seed):
  ancestors exact, X 1e-12, log-likelihood / filt / smo 1e-10, gradient 1e-9 * ||g||_inf (the SV tolerances).
- N = 2^20, T = 300: the same oracle with the tolerances DESIGN section 2 states at this N, and the Kalman filter.
- The fully adapted filter at N = 2^20 against the Kalman filter and the bootstrap filter.
- The SV model through this entry is bit-identical to pmmh_flps_sv_corr on the grid kernel.
- Bit reproducibility, kernel routing and the refusals.
"""
import ctypes

import numpy as np
import pytest

import golden_inputs as gi
from helpers import first_mismatch_step, relerr, to_time_major

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_SOFT_TIES, DIAG_KERNEL = 2, 4, 6
CHAIN, GRID = 3, 5
TILE_MAX = 7168   # particles of one grid-kernel tile (one CTA per SM)


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def _gpu_u(cuda_dev, nobs, n, seed, batch=1):
    """u [batch, nobs, n] (time-major) and rvr [batch, nobs] drawn on the device."""
    import torch
    g = torch.Generator(device=cuda_dev)
    g.manual_seed(seed)
    u = torch.randn((batch, nobs, n), dtype=torch.float64, device=cuda_dev, generator=g)
    rvr = torch.rand((batch, nobs), dtype=torch.float64, device=cuda_dev, generator=g)
    return u, rvr


def _flat(u):
    """device u [1, nobs, n] -> the reference's flat rvp[i + j * nobs]"""
    return np.ascontiguousarray(u[0].cpu().numpy().T).reshape(-1)


def _model_ws_bytes(n_obs, n, lag, batch):
    """pmmh_flps_model_workspace_bytes, or None where it refuses the sizes"""
    from pmmh_qn_b200 import _lib
    out = ctypes.c_size_t()
    rc = _lib.load().pmmh_flps_model_workspace_bytes(n_obs, n, lag, batch, ctypes.byref(out))
    return out.value if rc == 0 else None


@pytest.mark.parametrize("n,nobs,lag,seed", [(5000, 300, 10, 0), (4097, 150, 2, 1), (1 << 14, 120, 4, 1),
                                             (20000, 80, 10, 0), (20000, 60, 2, 1), (65536, 40, 10, 1),
                                             (65536, 50, 4, 0), (5003, 80, 10, 2), (20000, 60, 2, 2),
                                             (65536, 40, 4, 2), (4097, 100, 10, 3), (20000, 60, 2, 3)])
def test_linear_gaussian_on_the_grid_kernel_vs_generic_oracle(cuda_dev, n, nobs, lag, seed):
    import generic_pf as gp
    from pmmh_qn_b200 import _lib, kernels as K
    obs, params, rvr, rvp = gi.lg_inputs(n, nobs, seed)
    ref = gp.flps_generic(gp.LinearGaussian(params), obs, rvr, rvp, n, lag, dumps=True)
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, params, rvr[:nobs], to_time_major(rvp, n, nobs))
    out = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True)
    res = {k: v[0].cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    d = res["diag"]
    assert int(d[DIAG_KERNEL]) == GRID and int(d[DIAG_STATUS]) == 0, d
    step = first_mismatch_step(res["A"][1:], ref["A"][1:])
    if step is not None:
        # a resampling decision within the summation-order bound of a cumulative-weight tie may go the other way
        assert int(d[DIAG_SOFT_TIES]) > 0, "ancestors differ first at time %d without a counted tie" % (step + 1)
        assert relerr(res["X"][:step + 1], ref["X"][:step + 1]) <= 1e-12
        assert relerr(res["filt"][:step + 1], ref["filt"][:step + 1]) <= 1e-10
        return
    assert relerr(res["X"], ref["X"]) <= 1e-12
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"])
    assert relerr(res["filt"], ref["filt"]) <= 1e-10
    assert relerr(res["smo"], ref["smo"]) <= 1e-10
    assert relerr(res["traj"], ref["traj"]) <= 1e-12 and res["traj"][0] == ref["traj"][0] == 0.0
    g = res["gradient"]
    assert np.max(np.abs(g - ref["gradient"])) <= 1e-9 * np.max(np.abs(ref["gradient"]))
    assert np.all(g[3] == 0.0)


def test_linear_gaussian_headline_size(cuda_dev):
    """N = 2^20, T = 300 against the oracle (log-likelihood and filt 1e-10; smo and gradient 1e-4 * ||.||_inf: at this
    N a flipped neighbour moves the fixed-lag means by O(1/N), DESIGN section 2) and against the exact likelihood.
    Kalman bound: the N = 4096, T = 200 test allows 2.5 per estimate; the spread scales with sqrt(T / N), so
    2.5 * sqrt(4096 / 2^20) * sqrt(300 / 200) = 0.19 here."""
    import generic_pf as gp
    from pmmh_qn_b200 import _lib, kernels as K
    n, nobs, lag = 1 << 20, 301, 10
    params = np.array(gi.LG_PARAM_SETS[0])
    obs = gi.lg_obs(nobs, params)
    u, rvr = _gpu_u(cuda_dev, nobs, n, 21)
    obs_d, par_d = _dev(cuda_dev, obs, params)
    out = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr, u, lag=lag)
    res = {k: v[0].cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    assert int(res["diag"][DIAG_KERNEL]) == GRID and int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
    ref = gp.flps_generic(gp.LinearGaussian(params), obs, rvr[0].cpu().numpy(), _flat(u), n, lag)
    ll = float(res["log_like"])
    assert abs(ll - ref["log_like"]) <= 1e-10 * abs(ref["log_like"])
    assert relerr(res["filt"], ref["filt"]) <= 1e-10
    assert relerr(res["smo"], ref["smo"]) <= 1e-4
    assert np.max(np.abs(res["gradient"] - ref["gradient"])) <= 1e-4 * np.max(np.abs(ref["gradient"]))
    exact = gp.kalman_loglike(obs, *params[:3])
    assert abs(ll - exact) < 2.5 * np.sqrt(4096.0 / n) * np.sqrt(300.0 / 200.0), (ll, exact)


def test_fully_adapted_filter_at_2_20(cuda_dev):
    """log p(y_1) + the fully adapted estimate is consistent with the Kalman likelihood (the N = 4096 test's 0.5
    scaled by sqrt(4096 / N)); over 4 independent u its spread is smaller than the bootstrap filter's on the same
    data; its gradient rows are 0."""
    import generic_pf as gp
    from pmmh_qn_b200 import _lib, kernels as K
    n, nobs, lag, B = 1 << 20, 201, 10, 4
    params = np.array(gi.LG_PARAM_SETS[0])
    phi, sv, se = params[:3]
    obs = gi.lg_obs(nobs, params)
    exact = gp.kalman_loglike(obs, phi, sv, se)
    ll_y1 = gp.log_p_y1(obs, sv, se)
    obs_d, obs_s, par_d = _dev(cuda_dev, obs, obs[1:], params)                 # obs'[t] = obs[t + 1]
    fa, boot = [], []
    for r in range(B):
        u, rvr = _gpu_u(cuda_dev, nobs, n, 40 + r)
        b = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr, u, lag=lag)
        f = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA, obs_s, par_d, rvr[:, :nobs - 1].contiguous(),
                              u[:, :nobs - 1].contiguous(), lag=lag)
        for o in (b, f):
            assert int(o["diag"][0, DIAG_KERNEL]) == GRID and int(o["diag"][0, DIAG_STATUS]) == 0, o["diag"]
        assert np.all(f["gradient"].cpu().numpy() == 0.0)
        boot.append(float(b["log_like"][0]))
        fa.append(float(f["log_like"][0]) + ll_y1)
        del u
    fa, boot = np.array(fa), np.array(boot)
    assert np.all(np.abs(fa - exact) < 0.5 * np.sqrt(4096.0 / n)), (fa, exact)
    assert fa.std(ddof=1) < boot.std(ddof=1), (fa.std(ddof=1), boot.std(ddof=1))


@pytest.mark.parametrize("n", [1 << 14, 1 << 20])
def test_sv_through_the_model_entry_equals_the_sv_entry(cuda_dev, n):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    nobs, lag = 101, 10
    obs_d, par_d = _dev(cuda_dev, gi.sv_obs(nobs), np.array(gi.SV_PARAM_SETS[0]))
    u, rvr = _gpu_u(cuda_dev, nobs, n, 5)
    a = K.flps_model_corr(_lib.MODEL_SV_LEVERAGE, obs_d, par_d, rvr, u, lag=lag)
    K.set_sv_algorithm(0)
    b = K.flps_sv_corr(obs_d, par_d, rvr, u, lag=lag, compute_hessian=False)
    torch.cuda.synchronize()
    for o in (a, b):
        assert int(o["diag"][0, DIAG_KERNEL]) == GRID and int(o["diag"][0, DIAG_STATUS]) == 0, o["diag"]
    for k in ("log_like", "filt", "smo", "gradient", "traj"):
        assert torch.equal(a[k], b[k]), k


def test_linear_gaussian_at_2_20_is_bit_reproducible(cuda_dev):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    n, nobs = 1 << 20, 101
    params = np.array(gi.LG_PARAM_SETS[1])
    obs_d, par_d = _dev(cuda_dev, gi.lg_obs(nobs, params), params)
    u, rvr = _gpu_u(cuda_dev, nobs, n, 9)
    r1 = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr, u, lag=10)
    r2 = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr, u, lag=10)
    torch.cuda.synchronize()
    assert int(r1["diag"][0, DIAG_KERNEL]) == GRID and int(r1["diag"][0, DIAG_STATUS]) == 0
    for k in ("log_like", "filt", "smo", "gradient", "traj", "diag"):
        assert torch.equal(r1[k], r2[k]), k


def test_model_entry_routing_and_refusals(cuda_dev):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    sm = K.device_info()[0]
    params = np.array(gi.LG_PARAM_SETS[0])

    def call(n, nobs, lag, batch):
        obs_d, par_d = _dev(cuda_dev, gi.lg_obs(nobs, params), np.tile(params, (batch, 1)))
        u, rvr = _gpu_u(cuda_dev, nobs, n, 3, batch)
        try:
            out = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr, u, lag=lag)
        except _lib.PmmhError:
            return None
        torch.cuda.synchronize()
        return out["diag"][:, DIAG_KERNEL].cpu().numpy()

    cap = sm * TILE_MAX
    cases = [(4096, 40, 10, 3, CHAIN),          # the chain kernel keeps every shape it takes
             (1 << 16, 40, 10, 1, GRID),
             (cap, 30, 10, 1, GRID),            # the largest size one tile per SM holds
             (1 << 16, 40, 10, 2, None),        # batches of large problems
             (1 << 16, 40, 11, 1, None),        # lag above 10
             (1 << 16, 19, 10, 1, None),        # n_obs below 2 lag
             (cap + 1, 30, 10, 1, None)]        # above the grid kernel's capacity
    for n, nobs, lag, batch, want in cases:
        got = call(n, nobs, lag, batch)
        ws = _model_ws_bytes(nobs, n, lag, batch)
        if want is None:
            assert got is None and ws is None, (n, nobs, lag, batch, got, ws)
        else:
            assert got is not None and np.all(got == want) and ws, (n, nobs, lag, batch, got, ws)
