"""The fully adapted linear Gaussian filter (model id 2, csrc/pf_model.cuh) against its exact NumPy restatement
(oracle/generic_pf.py: LinearGaussianFullyAdapted through flps_generic), on the chain kernel (diag kernel 3) and
the grid kernel (diag kernel 5).  The Kalman-based tests of this model are statistical and the filter / smoother
entry comparisons run the same hooks on both sides; these pin the proposal gain and sd, child_range and logw_max
(phi < 0, phi = 0, a near unit root) operation for operation: ancestors exact, X and traj 1e-12, log-likelihood /
filt / smo 1e-10, gradient rows exactly 0 (the model has no score terms).

The observations handed to the device are the shifted series obs'[t] = obs[t + 1] and the restatement runs on the
same series, so both compute log p(y_2 .. y_T | y_1) and E[x_t | y_1 .. y_{t+1}].
"""
import numpy as np
import pytest

import golden_inputs as gi
from helpers import first_mismatch_step, relerr, to_time_major

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_SOFT_TIES, DIAG_KERNEL = 2, 4, 6
CHAIN, GRID = 3, 5
# the linear Gaussian sets (phi > 0, phi < 0, phi = 0) and a near unit root with a gain k = 0.0025
FA_PARAM_SETS = gi.LG_PARAM_SETS + [(0.999, 0.05, 1.0, 0.0)]


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def _fa_inputs(n, nobs, params, seed):
    """the shifted series obs[1:] of data simulated from params, rvr [nobs], rvp [nobs * N] (reference layout)"""
    obs = gi.lg_obs(nobs + 1, params)[1:]
    rvr, rvp = gi.split_particle(gi.sv_rvs(n, nobs, 500 + seed), nobs)
    return obs, rvr, rvp


def _fa_ref(obs, params, rvr, rvp, n, lag):
    import generic_pf as gp
    return gp.flps_generic(gp.LinearGaussianFullyAdapted(params), obs, rvr, rvp, n, lag, dumps=True)


def _check_exact(res, ref):
    """one problem's device outputs (NumPy) against the restatement, ancestors exact"""
    step = first_mismatch_step(res["A"][1:], ref["A"][1:])
    assert step is None, "ancestors differ first at time %d" % (step + 1)
    assert relerr(res["X"], ref["X"]) <= 1e-12
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"])
    assert relerr(res["filt"], ref["filt"]) <= 1e-10
    assert relerr(res["smo"], ref["smo"]) <= 1e-10
    assert relerr(res["traj"], ref["traj"]) <= 1e-12
    assert np.all(res["gradient"] == 0.0)


@pytest.mark.parametrize("lag", [2, 4, 10])
@pytest.mark.parametrize("n", [2, 3, 64, 1000, 4096])
def test_fully_adapted_on_the_chain_kernel_vs_restatement(cuda_dev, n, lag):
    """one batch of 5 problems with distinct parameters and data, each compared on its own"""
    from pmmh_qn_b200 import _lib, kernels as K
    nobs, B = 60, len(FA_PARAM_SETS)
    cases = [_fa_inputs(n, nobs, p, b) for b, p in enumerate(FA_PARAM_SETS)]
    obs = np.stack([c[0] for c in cases])
    rvr = np.stack([c[1] for c in cases])
    u = np.stack([to_time_major(c[2], n, nobs) for c in cases])
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, np.array(FA_PARAM_SETS), rvr, u)
    out = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True)
    res = {k: v.cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    assert np.all(res["diag"][:, DIAG_KERNEL] == CHAIN) and np.all(res["diag"][:, DIAG_STATUS] == 0), res["diag"]
    for b, p in enumerate(FA_PARAM_SETS):
        ref = _fa_ref(obs[b], p, rvr[b], cases[b][2], n, lag)
        _check_exact({k: v[b] for k, v in res.items()}, ref)


@pytest.mark.parametrize("pset", range(len(FA_PARAM_SETS)))
@pytest.mark.parametrize("lag", [2, 10])
@pytest.mark.parametrize("n", [4097, 5003, 1 << 14, 65536])
def test_fully_adapted_on_the_grid_kernel_vs_restatement(cuda_dev, n, lag, pset):
    from pmmh_qn_b200 import _lib, kernels as K
    nobs, params = 50, FA_PARAM_SETS[pset]
    obs, rvr, rvp = _fa_inputs(n, nobs, params, pset)
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, np.array(params), rvr, to_time_major(rvp, n, nobs))
    out = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True)
    res = {k: v[0].cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    d = res["diag"]
    assert int(d[DIAG_KERNEL]) == GRID and int(d[DIAG_STATUS]) == 0, d
    ref = _fa_ref(obs, params, rvr, rvp, n, lag)
    step = first_mismatch_step(res["A"][1:], ref["A"][1:])
    if step is not None:
        # a resampling decision within the summation-order bound of a cumulative-weight tie may go the other way
        assert int(d[DIAG_SOFT_TIES]) > 0, "ancestors differ first at time %d without a counted tie" % (step + 1)
        assert relerr(res["X"][:step + 1], ref["X"][:step + 1]) <= 1e-12
        assert relerr(res["filt"][:step + 1], ref["filt"][:step + 1]) <= 1e-10
        assert np.all(res["gradient"] == 0.0)
        return
    _check_exact(res, ref)


def test_fully_adapted_on_the_grid_kernel_at_2_20(cuda_dev):
    """N = 2^20, T = 40, phi < 0: log-likelihood and filt 1e-10; smo 1e-4 (at this N a flipped neighbour moves the
    fixed-lag means by O(1/N), DESIGN section 2)."""
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    n, nobs, lag = 1 << 20, 40, 10
    params = gi.LG_PARAM_SETS[2]
    obs = gi.lg_obs(nobs + 1, params)[1:]
    g = torch.Generator(device=cuda_dev)
    g.manual_seed(77)
    u = torch.randn((1, nobs, n), dtype=torch.float64, device=cuda_dev, generator=g)
    rvr = torch.rand((1, nobs), dtype=torch.float64, device=cuda_dev, generator=g)
    obs_d, par_d = _dev(cuda_dev, obs, np.array(params))
    out = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA, obs_d, par_d, rvr, u, lag=lag)
    res = {k: v[0].cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    assert int(res["diag"][DIAG_KERNEL]) == GRID and int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
    import generic_pf as gp
    rvp = np.ascontiguousarray(u[0].cpu().numpy().T).reshape(-1)
    ref = gp.flps_generic(gp.LinearGaussianFullyAdapted(params), obs, rvr[0].cpu().numpy(), rvp, n, lag)
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"])
    assert relerr(res["filt"], ref["filt"]) <= 1e-10
    assert relerr(res["smo"], ref["smo"]) <= 1e-4
    assert np.all(res["gradient"] == 0.0)
