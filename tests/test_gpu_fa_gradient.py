"""Model id 4 (the fully adapted linear Gaussian filter with a fixed-lag gradient, csrc/pf_model.cuh) on the chain
kernel (diag kernel 3), the one-problem grid kernel and the team grid kernel (diag kernel 5):

- against its operation-for-operation restatement (tests/fa_gradient_oracle.py flps_fa_grad): ancestors
  exact, X / traj 1e-12, log-likelihood / filt / smo 1e-10, gradient per slot 1e-9 of its largest entry;
- everything model 2 outputs (filt, smo, log_like, traj, diag, X, A) bit-identical to model 2's on the same inputs;
  each problem of a team batch bit-identical to its one-problem run; the filter entries take id 4 as id 2;
- compute_hessian with id 4 is refused, and so is the unassigned id 3.
The observations handed to the device are the shifted series obs' = obs[1:], as for model 2."""
import numpy as np
import pytest

import golden_inputs as gi
from helpers import first_mismatch_step, relerr, to_time_major

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_SOFT_TIES, DIAG_KERNEL = 2, 4, 6
CHAIN, GRID = 3, 5
FA, FAG = 2, 4
# the linear Gaussian sets (phi > 0, phi < 0, phi = 0) and a near unit root with a gain k = 0.0025
FA_PARAM_SETS = gi.LG_PARAM_SETS + [(0.999, 0.05, 1.0, 0.0)]
SHARED = ("filt", "smo", "log_like", "traj", "diag", "X", "A")


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def _inputs(n, nobs, params, seed):
    """the shifted series obs[1:] of data simulated from params, rvr [nobs], rvp [nobs * N] (reference layout)"""
    obs = gi.lg_obs(nobs + 1, params)[1:]
    rvr, rvp = gi.split_particle(gi.sv_rvs(n, nobs, 600 + seed), nobs)
    return obs, rvr, rvp


def _ref(obs, params, rvr, rvp, n, lag):
    import fa_gradient_oracle as fo
    return fo.flps_fa_grad(params, obs, rvr, rvp, n, lag, dumps=True)


def _np(out, b=None):
    return {k: (v.cpu().numpy() if b is None else v[b].cpu().numpy()) for k, v in out.items() if not k.startswith("_")}


def _check_exact(res, ref):
    """one problem's device outputs (NumPy) against the restatement, ancestors exact"""
    step = first_mismatch_step(res["A"][1:], ref["A"][1:])
    assert step is None, "ancestors differ first at time %d" % (step + 1)
    assert relerr(res["X"], ref["X"]) <= 1e-12
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"])
    assert relerr(res["filt"], ref["filt"]) <= 1e-10
    assert relerr(res["smo"], ref["smo"]) <= 1e-10
    assert relerr(res["traj"], ref["traj"]) <= 1e-12
    g, gr = res["gradient"], ref["gradient"]
    assert np.all(g[3] == 0.0)
    assert np.max(np.abs(g - gr)) <= 1e-9 * np.max(np.abs(gr)), np.max(np.abs(g - gr)) / np.max(np.abs(gr))


def _same(a, b, keys=SHARED):
    for k in keys:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("lag", [2, 4, 10])
@pytest.mark.parametrize("n", [2, 3, 64, 1000, 4096])
def test_chain_kernel_vs_restatement_and_model_2(cuda_dev, n, lag):
    """one batch of 5 problems with distinct parameters and data, each compared on its own; the same batch as model 2"""
    from pmmh_qn_b200 import kernels as K
    nobs = 60
    cases = [_inputs(n, nobs, p, b) for b, p in enumerate(FA_PARAM_SETS)]
    obs = np.stack([c[0] for c in cases])
    rvr = np.stack([c[1] for c in cases])
    u = np.stack([to_time_major(c[2], n, nobs) for c in cases])
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, np.array(FA_PARAM_SETS), rvr, u)
    res = _np(K.flps_model_corr(FAG, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True))
    assert np.all(res["diag"][:, DIAG_KERNEL] == CHAIN) and np.all(res["diag"][:, DIAG_STATUS] == 0), res["diag"]
    for b, p in enumerate(FA_PARAM_SETS):
        _check_exact({k: v[b] for k, v in res.items()}, _ref(obs[b], p, rvr[b], cases[b][2], n, lag))
    _same(res, _np(K.flps_model_corr(FA, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True)))


@pytest.mark.parametrize("lag", [2, 4, 10])
def test_shortest_series_vs_restatement(cuda_dev, lag):
    """n_obs = lag + 1 on the chain kernel (main loop: slots 0 and 1, the tail the rest) and n_obs = 2 lag on the grid
    kernel, set 1 (phi 0.95)"""
    from pmmh_qn_b200 import kernels as K
    params = FA_PARAM_SETS[1]
    for n, nobs, kernel in ((1000, lag + 1, CHAIN), (4097, 2 * lag, GRID)):
        obs, rvr, rvp = _inputs(n, nobs, params, 90 + lag)
        obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, np.array([params]), rvr[None], to_time_major(rvp, n, nobs)[None])
        res = _np(K.flps_model_corr(FAG, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True), 0)
        assert int(res["diag"][DIAG_KERNEL]) == kernel and int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
        _check_exact(res, _ref(obs, params, rvr, rvp, n, lag))


@pytest.mark.parametrize("pset", [0, 2, 4])
@pytest.mark.parametrize("lag", [2, 10])
@pytest.mark.parametrize("n", [4097, 5003, 1 << 14, 65536])
def test_grid_kernel_vs_restatement(cuda_dev, n, lag, pset):
    from pmmh_qn_b200 import kernels as K
    nobs, params = 50, FA_PARAM_SETS[pset]
    obs, rvr, rvp = _inputs(n, nobs, params, pset)
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, np.array(params), rvr, to_time_major(rvp, n, nobs))
    res = _np(K.flps_model_corr(FAG, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True), 0)
    d = res["diag"]
    assert int(d[DIAG_KERNEL]) == GRID and int(d[DIAG_STATUS]) == 0, d
    ref = _ref(obs, params, rvr, rvp, n, lag)
    step = first_mismatch_step(res["A"][1:], ref["A"][1:])
    if step is not None:
        # a resampling decision within the summation-order bound of a cumulative-weight tie may go the other way
        assert int(d[DIAG_SOFT_TIES]) > 0, "ancestors differ first at time %d without a counted tie" % (step + 1)
        assert relerr(res["X"][:step + 1], ref["X"][:step + 1]) <= 1e-12
        assert relerr(res["filt"][:step + 1], ref["filt"][:step + 1]) <= 1e-10
        return
    _check_exact(res, ref)


def test_grid_kernel_at_2_20_vs_restatement(cuda_dev):
    """N = 2^20, T = 40, phi < 0: log-likelihood and filt 1e-10; smo and the gradient slots 1e-4 of their largest entry
    (at this N a flipped neighbour moves the fixed-lag means by O(1/N), DESIGN section 2), exact when no ancestor
    differs."""
    import torch
    import fa_gradient_oracle as fo
    from pmmh_qn_b200 import kernels as K
    n, nobs, lag = 1 << 20, 40, 10
    params = gi.LG_PARAM_SETS[2]
    obs = gi.lg_obs(nobs + 1, params)[1:]
    g = torch.Generator(device=cuda_dev)
    g.manual_seed(78)
    u = torch.randn((1, nobs, n), dtype=torch.float64, device=cuda_dev, generator=g)
    rvr = torch.rand((1, nobs), dtype=torch.float64, device=cuda_dev, generator=g)
    obs_d, par_d = _dev(cuda_dev, obs, np.array(params))
    res = _np(K.flps_model_corr(FAG, obs_d, par_d, rvr, u, lag=lag, store_history=True), 0)
    assert int(res["diag"][DIAG_KERNEL]) == GRID and int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
    rvp = np.ascontiguousarray(u[0].cpu().numpy().T).reshape(-1)
    ref = fo.flps_fa_grad(params, obs, rvr[0].cpu().numpy(), rvp, n, lag, dumps=True)
    if first_mismatch_step(res["A"][1:], ref["A"][1:]) is None:
        _check_exact(res, ref)
        return
    assert int(res["diag"][DIAG_SOFT_TIES]) > 0
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"])
    assert relerr(res["filt"], ref["filt"]) <= 1e-10
    assert relerr(res["smo"], ref["smo"]) <= 1e-4
    assert relerr(res["gradient"], ref["gradient"]) <= 1e-4


def test_one_problem_grid_kernel_and_team_batch_share_model_2_and_each_other(cuda_dev):
    """N = 2^14, 3 problems: model 4's shared outputs and history equal model 2's on the one-problem grid kernel and in
    a team batch, and each batch problem (gradient included) equals its one-problem run."""
    from pmmh_qn_b200 import kernels as K
    n, nobs, lag = 1 << 14, 40, 10
    sets = [0, 2, 4]
    cases = [_inputs(n, nobs, FA_PARAM_SETS[s], 50 + s) for s in sets]
    obs = np.stack([c[0] for c in cases])
    par = np.array([FA_PARAM_SETS[s] for s in sets])
    rvr = np.stack([c[1] for c in cases])
    u = np.stack([to_time_major(c[2], n, nobs) for c in cases])
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, par, rvr, u)
    b3 = _np(K.flps_model_batch_corr(FAG, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True))
    b2 = _np(K.flps_model_batch_corr(FA, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True))
    assert np.all(b3["diag"][:, DIAG_KERNEL] == GRID) and np.all(b3["diag"][:, DIAG_STATUS] == 0)
    _same(b3, b2)
    assert np.all(b2["gradient"] == 0.0) and np.any(b3["gradient"] != 0.0)
    for b in range(len(sets)):
        one = [_np(K.flps_model_corr(m, obs_d[b], par_d[b:b + 1], rvr_d[b:b + 1], u_d[b:b + 1], lag=lag,
                                     store_history=True), 0) for m in (FAG, FA)]
        _same(one[0], one[1])
        _same({k: v[b] for k, v in b3.items()}, one[0], SHARED + ("gradient",))


@pytest.mark.parametrize("n", [1000, 1 << 14])
def test_filter_entries_take_id_3_as_id_2(cuda_dev, n):
    from pmmh_qn_b200 import kernels as K
    nobs, B = 40, 3 if n <= 4096 else 2
    cases = [_inputs(n, nobs, FA_PARAM_SETS[b], 70 + b) for b in range(B)]
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, np.stack([c[0] for c in cases]), np.array(FA_PARAM_SETS[:B]),
                                    np.stack([c[1] for c in cases]),
                                    np.stack([to_time_major(c[2], n, nobs) for c in cases]))
    keys = ("filt", "log_like", "traj", "diag", "X", "A")
    if n <= 4096:
        _same(_np(K.filter_model_corr(FAG, obs_d, par_d, rvr_d, u_d, store_history=True)),
              _np(K.filter_model_corr(FA, obs_d, par_d, rvr_d, u_d, store_history=True)), keys)
    else:
        _same(_np(K.filter_model_corr(FAG, obs_d[0], par_d[:1], rvr_d[:1], u_d[:1], store_history=True)),
              _np(K.filter_model_corr(FA, obs_d[0], par_d[:1], rvr_d[:1], u_d[:1], store_history=True)), keys)
    _same(_np(K.filter_model_batch_corr(FAG, obs_d, par_d, rvr_d, u_d, store_history=True)),
          _np(K.filter_model_batch_corr(FA, obs_d, par_d, rvr_d, u_d, store_history=True)), keys)


def test_hessian_with_id_4_and_the_unassigned_id_3_are_refused(cuda_dev):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    n, nobs = 1 << 14, 40
    obs, rvr, rvp = _inputs(n, nobs, FA_PARAM_SETS[0], 0)
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, np.array([FA_PARAM_SETS[0]]), rvr[None], to_time_major(rvp, n, nobs)[None])
    with pytest.raises(_lib.PmmhError):
        K.flps_model_batch_corr(FAG, obs_d, par_d, rvr_d, u_d, lag=10, compute_hessian=1)
    for entry in (K.flps_model_corr, K.flps_model_batch_corr):   # id 3 is unassigned
        with pytest.raises(_lib.PmmhError):
            entry(3, obs_d, par_d, rvr_d, u_d, lag=10)
    for entry in (K.filter_model_corr, K.filter_model_batch_corr):
        with pytest.raises(_lib.PmmhError):
            entry(3, obs_d, par_d, rvr_d, u_d)
    torch.cuda.synchronize()
