"""Model id 6 (the fully adapted linear Gaussian filter with a fixed-lag Hessian, csrc/pf_model.cuh) on the grid kernel:

- hess1 / hess2 against the restatement (tests/fa_hessian_oracle.py predictive_hessian) replayed on the kernel's own
  history, 1e-10 of the largest entry;
- every output model 4 has is bit-identical to model 4's, on flps_model_corr (chain and grid kernels) and on
  flps_model_batch_corr with compute_hessian 0 and 1; the filter entries run model 2's filter;
- team batches bit-identical to one-problem runs, hess1 / hess2 included;
- the summed hess1 and hess1 + hess2 - g g' against the exact Kalman quantities over independent replicates;
- compute_hessian = 2 is refused; the estimator LinearGaussianParticleMethodsCUDA(hessian=True) publishes the entry's
  Hessian estimate.
The observations handed to the device are the shifted series obs' = obs[1:], as for models 2 and 4."""
import numpy as np
import pytest

import fa_hessian_oracle as fh
import generic_pf as gp
import golden_inputs as gi
from helpers import to_time_major

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_KERNEL = 2, 6
CHAIN, GRID = 3, 5
FA, FAG, FAH = 2, 4, 6
SHARED = ("filt", "smo", "log_like", "gradient", "traj", "diag", "X", "A")


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def _np(out, b=None):
    return {k: (v.cpu().numpy() if b is None else v[b].cpu().numpy()) for k, v in out.items() if not k.startswith("_")}


def _inputs(cuda_dev, n, nobs, params, seed, batch=1):
    """the shifted series of data simulated from params, rvr [B, nobs], u [B, nobs, N] (device); obs' [nobs] (host)"""
    import torch
    obs = gi.lg_obs(nobs + 1, params, seed=300 + seed)[1:]
    g = torch.Generator(device=cuda_dev)
    g.manual_seed(seed)
    u = torch.randn((batch, nobs, n), dtype=torch.float64, device=cuda_dev, generator=g)
    rvr = torch.rand((batch, nobs), dtype=torch.float64, device=cuda_dev, generator=g)
    par = torch.from_numpy(np.tile(np.asarray(params, dtype=np.float64), (batch, 1))).to(cuda_dev)
    return obs, _dev(cuda_dev, obs)[0], par, rvr, u


def _weights(params, obs, X):
    m = gp.LinearGaussianFullyAdapted(params)
    W = np.zeros_like(X)
    W[0] = 1.0 / X.shape[1]
    for i in range(1, X.shape[0]):
        lw = m.logw(X[i], obs[i])
        sh = np.exp(lw - np.max(lw))
        W[i] = sh / np.sum(sh)
    return W


@pytest.mark.parametrize("lag", [2, 10])
@pytest.mark.parametrize("n", [256, 8192, 1 << 14, 1 << 17])
def test_hessian_vs_restatement_on_the_kernels_history(cuda_dev, n, lag):
    """n_obs = 40 (set 0) and the shortest series n_obs = 2 lag (set 1)"""
    from pmmh_qn_b200 import kernels as K
    for nobs, pset in ((40, 0), (2 * lag, 1)):
        params = gi.LG_PARAM_SETS[pset]
        obs, obs_d, par, rvr, u = _inputs(cuda_dev, n, nobs, params, 17 * lag + pset)
        res = _np(K.flps_model_batch_corr(FAH, obs_d, par, rvr, u, lag=lag, compute_hessian=1, store_history=True), 0)
        assert int(res["diag"][DIAG_KERNEL]) == GRID and int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
        X, A = res["X"], res["A"].astype(np.int64)
        h1, h2 = fh.predictive_hessian(fh.LinearGaussianFullyAdaptedHess(params), obs, X, A, _weights(params, obs, X), lag)
        for got, want in ((res["hess1"], h1), (res["hess2"], h2)):
            assert np.max(np.abs(got - want)) <= 1e-10 * np.max(np.abs(want)), (n, lag, nobs, got, want)
        assert np.all(res["hess1"][3] == 0.0) and np.all(res["hess2"][:, 3] == 0.0)
        assert np.array_equal(res["hess1"], res["hess1"].T) and np.array_equal(res["hess2"], res["hess2"].T)


@pytest.mark.parametrize("n", [1000, 1 << 14])
def test_outputs_bit_identical_to_model_4(cuda_dev, n):
    """flps_model_corr (chain kernel at 1000 particles, 3 problems; grid kernel at 2^14) and flps_model_batch_corr
    with compute_hessian 0 and 1; the filter entries give model 2's filter"""
    from pmmh_qn_b200 import kernels as K
    nobs, lag = 40, 10
    B = 3 if n <= 4096 else 1
    _, obs_d, par, rvr, u = _inputs(cuda_dev, n, nobs, gi.LG_PARAM_SETS[0], 5, batch=B)
    one = [_np(K.flps_model_corr(m, obs_d, par, rvr, u, lag=lag, store_history=True)) for m in (FAG, FAH)]
    assert np.all(one[0]["diag"][:, DIAG_KERNEL] == (CHAIN if n <= 4096 else GRID))
    for k in SHARED:
        assert np.array_equal(one[0][k], one[1][k]), k
    b4 = _np(K.flps_model_batch_corr(FAG, obs_d, par, rvr, u, lag=lag, store_history=True))
    for hess in (0, 1):
        b6 = _np(K.flps_model_batch_corr(FAH, obs_d, par, rvr, u, lag=lag, compute_hessian=hess, store_history=True))
        for k in SHARED:
            assert np.array_equal(b4[k], b6[k]), (hess, k)
        assert ("hess1" in b6) == bool(hess)
    keys = ("filt", "log_like", "traj", "diag", "X", "A")
    f2, f6 = (_np(K.filter_model_corr(m, obs_d, par, rvr, u, store_history=True)) for m in (FA, FAH))
    for k in keys:
        assert np.array_equal(f2[k], f6[k]), k


@pytest.mark.parametrize("n,batch", [(1 << 14, 20), (1 << 16, 5)])
def test_team_batch_bit_identical_to_one_problem_runs(cuda_dev, n, batch):
    from pmmh_qn_b200 import kernels as K
    nobs, lag = 40, 10
    sets = [b % 4 for b in range(batch)]
    import torch
    cases = [_inputs(cuda_dev, n, nobs, gi.LG_PARAM_SETS[s], 900 + b) for b, s in enumerate(sets)]
    obs_d = torch.stack([c[1] for c in cases])
    par, rvr, u = (torch.cat([c[i] for c in cases]) for i in (2, 3, 4))
    bt = _np(K.flps_model_batch_corr(FAH, obs_d, par, rvr, u, lag=lag, compute_hessian=1))
    assert np.all(bt["diag"][:, DIAG_KERNEL] == GRID) and np.all(bt["diag"][:, DIAG_STATUS] == 0)
    for b in range(batch):
        one = _np(K.flps_model_batch_corr(FAH, obs_d[b], par[b:b + 1], rvr[b:b + 1], u[b:b + 1], lag=lag,
                                          compute_hessian=1), 0)
        for k in ("filt", "smo", "log_like", "gradient", "traj", "diag", "hess1", "hess2"):
            assert np.array_equal(bt[k][b], one[k]), (b, k)


def test_hessian_against_kalman(cuda_dev):
    """n' = 20, lag 10, phi = 0.5 (the CPU set-up of test_fa_hessian_reference.py), 72 replicates at N = 2^14 in one
    team batch: the summed hess1 against the exact targets and hess1 + hess2 - g g' against the exact Hessian of the
    Kalman log-likelihood, |z| <= 5 per entry."""
    import torch
    from pmmh_qn_b200 import kernels as K
    params, nprime, lag, n, k = (0.5, 0.6, 0.4, 0.0), 20, 10, 1 << 14, 72
    obs = gi.lg_obs(nprime + 1, params, seed=4242)
    g = torch.Generator(device=cuda_dev)
    g.manual_seed(2024)
    u = torch.randn((k, nprime, n), dtype=torch.float64, device=cuda_dev, generator=g)
    rvr = torch.rand((k, nprime), dtype=torch.float64, device=cuda_dev, generator=g)
    par = torch.from_numpy(np.tile(np.asarray(params, dtype=np.float64), (k, 1))).to(cuda_dev)
    out = _np(K.flps_model_batch_corr(FAH, _dev(cuda_dev, obs[1:])[0], par, rvr, u, lag=lag, compute_hessian=1))
    assert np.all(out["diag"][:, DIAG_STATUS] == 0)
    est = np.array([fh.hessian_estimate({kk: out[kk][b] for kk in ("gradient", "hess1", "hess2")}) for b in range(k)])
    h1 = out["hess1"][:, :3, :3]
    for name, reps, exact in (("hess1", h1, fh.hess1_targets(obs, *params[:3], lag).sum(axis=0)),
                              ("hessian", est, fh.kalman_hessian(obs, *params[:3]))):
        s = reps.std(axis=0, ddof=1)
        live = s > 0.0
        z = (reps.mean(axis=0) - exact)[live] / (s[live] / np.sqrt(k))
        print(name, "exact", np.round(exact, 3).tolist(), "z", np.round(z, 2).tolist())
        assert np.all(np.abs(z) <= 5.0), (name, z)


def test_compute_hessian_2_is_refused(cuda_dev):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    _, obs_d, par, rvr, u = _inputs(cuda_dev, 1 << 14, 40, gi.LG_PARAM_SETS[0], 3)
    with pytest.raises(_lib.PmmhError):
        K._model_corr("flps_model_batch", FAH, obs_d, par, rvr, u, 10, 2, False, None)
    torch.cuda.synchronize()


class _LGSS(object):
    short_name = 'lgss'

    def __init__(self, obs, params):
        self.obs = np.asarray(obs, dtype=np.float64).reshape(-1, 1)
        self.no_obs = self.obs.shape[0] - 1
        self.params = {'phi': float(params[0]), 'sigma_v': float(params[1]), 'sigma_e': float(params[2])}
        self.no_params = 3
        self.params_to_estimate = ('phi', 'sigma_v', 'sigma_e')
        self.params_to_estimate_idx = np.arange(3)
        self.no_params_to_estimate = 3
        self.using_gradients = True
        self.using_hessians = True

    def get_all_params(self):
        return np.array([self.params[k] for k in self.params])

    def log_prior_gradient(self):
        return {k: 0.0 for k in self.params}

    def log_prior_hessian(self):
        return {k: 0.0 for k in self.params}


def test_estimator_publishes_the_entrys_hessian(cuda_dev):
    from pmmh_qn_b200 import LinearGaussianParticleMethodsCUDA
    from pmmh_qn_b200 import kernels as K
    n, nobs, lag = 1000, 50, 6
    params = gi.LG_PARAM_SETS[0]
    obs = gi.lg_obs(nobs, params, seed=5000)
    model = _LGSS(obs, params)
    rvs = gi.sv_rvs(n, nobs - 1, 31)
    rvr, rvp = gi.split_particle(rvs, nobs - 1)
    obs_d, par, rvr_d, u = _dev(cuda_dev, obs[1:], np.array([params]), rvr[None], to_time_major(rvp, n, nobs - 1)[None])
    ref = _np(K.flps_model_batch_corr(FAH, obs_d, par, rvr_d, u, lag=lag, compute_hessian=1), 0)
    want = fh.hessian_estimate(ref)
    est = LinearGaussianParticleMethodsCUDA(model, n, fixed_lag=lag, hessian=True)
    assert est.smoother(model, rvs={'rvs': rvs})
    r = est.results
    assert est.settings['estimate_hessian']
    assert np.array_equal(r['hessian_internal'], want) and np.array_equal(r['hessian_internal_noprior'], want)
    assert np.array_equal(r['gradient_internal'], ref["gradient"][:3].sum(axis=1))
    assert abs(r['log_like'] - (float(ref["log_like"]) + gp.log_p_y1(obs, params[1], params[2]))) <= 1e-12 * abs(r['log_like'])
    assert not LinearGaussianParticleMethodsCUDA(model, n, fixed_lag=lag).smoother(model, rvs={'rvs': rvs})
