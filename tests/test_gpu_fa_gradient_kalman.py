"""Model id 4's gradient on the GPU against the exact fixed-lag Kalman targets (tests/fa_gradient_oracle.py fa_gradient_targets),
over replicate u's with fixed seeds, with the thresholds of test_gpu_model_kalman.py: per slot RMS z <= 1.5 and
max |z| <= 6; summed |mean - exact| <= 4.5 s / sqrt(K), s at most twice the restatement's spread at the same N.  Also
the estimator LinearGaussianParticleMethodsCUDA: its results are the entry's, and a correlated PMMH run completes.
The z statistics are printed (pytest -s)."""
import numpy as np
import pytest

import fa_gradient_oracle as fo
import generic_pf as gp
import golden_inputs as gi

pytestmark = pytest.mark.gpu

Z_RMS, Z_MAX, Z_SUM, S_CEIL = 1.5, 6.0, 4.5, 2.0
LG, FAG = 1, 4


def _obs(nobs, pset):
    return gi.lg_obs(nobs, gi.LG_PARAM_SETS[pset], seed=5000 + pset)


def _u(cuda_dev, k, nobs, n, seed):
    import torch
    g = torch.Generator(device=cuda_dev)
    g.manual_seed(seed)
    u = torch.randn((k, nobs, n), dtype=torch.float64, device=cuda_dev, generator=g)
    rvr = torch.rand((k, nobs), dtype=torch.float64, device=cuda_dev, generator=g)
    return u, rvr


def _zslots(name, reps, exact):
    """A slot every replicate gives the same value (the phi term of the pair (x_0, x_1): x_0 = 0) must equal the
    target; the others enter the z statistics."""
    reps = np.asarray(reps)
    k = reps.shape[0]
    s = reps.std(axis=0, ddof=1)
    flat = s == 0.0
    assert np.all(np.abs(reps[0, flat] - exact[flat]) <= 1e-12 * np.maximum(np.abs(exact[flat]), 1.0)), name
    z = (reps.mean(axis=0) - exact)[~flat] / (s[~flat] / np.sqrt(k))
    rms, zmax = float(np.sqrt(np.mean(z * z))), float(np.max(np.abs(z)))
    print("%-44s K %3d slots %4d  RMS z %.2f  max |z| %.2f" % (name, k, z.size, rms, zmax))
    assert rms <= Z_RMS and zmax <= Z_MAX, "%s: RMS z %.2f, max |z| %.2f at slot %d" % (name, rms, zmax, int(np.argmax(np.abs(z))))


def _cpu_sd(obs, params, n, lag, runs=16):
    """Spread of the restatement's summed gradient at N = n (model 4, on obs[1:])."""
    o = obs[1:]
    tot = []
    for seed in range(runs):
        rvr, rvp = gi.split_particle(gi.sv_rvs(n, len(o), 900 + seed), len(o))
        tot.append(fo.flps_fa_grad(params, o, rvr, rvp, n, lag)["gradient"].sum(axis=1)[:3])
    return np.std(tot, axis=0, ddof=1)


def _zsum(name, grads, exact, ceiling=None):
    tot = np.asarray(grads)[:, :3].sum(axis=2)
    k = tot.shape[0]
    mean, s = tot.mean(axis=0), tot.std(axis=0, ddof=1)
    z = (mean - exact) / (s / np.sqrt(k))
    print("%-44s K %3d summed z %s  s %s%s" % (name, k, np.round(z, 2), np.round(s, 3),
                                               "" if ceiling is None else "  ceiling %s" % np.round(ceiling, 3)))
    assert np.all(np.abs(z) <= Z_SUM), "%s: summed gradient %s vs exact %s (z %s)" % (name, mean, exact, z)
    if ceiling is not None:
        assert np.all(s <= ceiling), "%s: spread %s above %s" % (name, s, ceiling)
    return s


def _check(name, out, obs, params, lag, rows=None, ceiling_n=None):
    phi, sv, se = params[:3]
    rows = slice(None) if rows is None else rows
    grad = out["gradient"].cpu().numpy()[rows]
    assert int(out["diag"][:, 2].max()) == 0
    tg = fo.fa_gradient_targets(obs, phi, sv, se, lag)
    assert np.all(grad[:, 3] == 0.0)
    for q, p in enumerate(("phi", "sigma_v", "sigma_e")):
        _zslots("%s gradient %s" % (name, p), grad[:, q], tg["grad"][q])
    ceil = None if ceiling_n is None else S_CEIL * _cpu_sd(obs, params, ceiling_n, lag)
    _zsum(name, grad, tg["grad_sum"], ceil)


def _run(cuda_dev, entry, model, obs, params, n, lag, k, seed):
    import torch
    o = obs[1:] if model == FAG else obs
    u, rvr = _u(cuda_dev, k, len(obs), n, seed)
    u, rvr = u[:, :len(o)].contiguous(), rvr[:, :len(o)].contiguous()
    par = torch.from_numpy(np.tile(np.asarray(params, dtype=np.float64), (k, 1))).to(cuda_dev)
    return entry(model, torch.from_numpy(np.ascontiguousarray(o)).to(cuda_dev), par, rvr, u, lag=lag)


@pytest.mark.parametrize("n,nobs,lag,pset", [(4096, 61, 10, 0), (4096, 61, 2, 2), (257, 61, 2, 3), (257, 31, 4, 0)])
def test_chain_kernel_against_exact_targets(cuda_dev, n, nobs, lag, pset):
    """64 replicates at N = 4096, 16 at N = 257.  (The shortest series are pinned to the restatement in
    test_gpu_fa_gradient.py: at n_obs = lag + 1 nearly every slot is read under the final weights, the slots' errors
    are correlated (|corr| up to 0.7 in the restatement, set 1) and their RMS z is no longer that of independent
    slots.)"""
    from pmmh_qn_b200 import kernels as K
    params = gi.LG_PARAM_SETS[pset]
    obs = _obs(nobs, pset)
    out = _run(cuda_dev, K.flps_model_corr, FAG, obs, params, n, lag, 64 if n >= 4096 else 16, seed=20 * pset + lag)
    assert int(out["diag"][:, 6].min()) == 3
    _check("chain m3 N %d T %d lag %d set %d" % (n, nobs, lag, pset), out, obs, params, lag, ceiling_n=n)


def test_chain_kernel_mixed_parameter_batch(cuda_dev):
    """One batch of 64 problems cycling through the four parameter sets, each with its own series."""
    import torch
    from pmmh_qn_b200 import kernels as K
    k, n, nobs, lag = 64, 4096, 51, 4
    sets = [b % 4 for b in range(k)]
    obs = np.stack([_obs(nobs, s) for s in sets])
    params = np.array([gi.LG_PARAM_SETS[s] for s in sets], dtype=np.float64)
    u, rvr = _u(cuda_dev, k, nobs - 1, n, seed=91)
    out = K.flps_model_corr(FAG, torch.from_numpy(np.ascontiguousarray(obs[:, 1:])).to(cuda_dev),
                            torch.from_numpy(params).to(cuda_dev), rvr, u, lag=lag)
    for s in range(4):
        _check("chain mixed lag %d set %d" % (lag, s), out, obs[s], gi.LG_PARAM_SETS[s], lag, rows=np.arange(s, k, 4))


@pytest.mark.parametrize("nobs,lag,pset", [(61, 10, 1), (61, 2, 0), (21, 10, 2)])
def test_team_grid_kernel_against_exact_targets(cuda_dev, nobs, lag, pset):
    """flps_model_batch_corr, 36 replicates at N = 2^14 (two waves on a 148-SM B200)."""
    from pmmh_qn_b200 import kernels as K
    params = gi.LG_PARAM_SETS[pset]
    obs = _obs(nobs, pset)
    out = _run(cuda_dev, K.flps_model_batch_corr, FAG, obs, params, 1 << 14, lag, 36, seed=330 + 10 * pset + lag)
    assert int(out["diag"][:, 6].min()) == 5
    _check("team grid m3 N 2^14 T %d lag %d set %d" % (nobs, lag, pset), out, obs, params, lag,
           ceiling_n=(1 << 14) if nobs <= 21 else None)


def test_one_problem_grid_kernel_summed_gradient(cuda_dev):
    """N = 2^20, lag 10, six replicates: the summed gradient."""
    from pmmh_qn_b200 import kernels as K
    n, nobs, lag, k, pset = 1 << 20, 41, 10, 6, 0
    params = gi.LG_PARAM_SETS[pset]
    phi, sv, se = params[:3]
    obs = _obs(nobs, pset)
    grads = []
    for r in range(k):
        out = _run(cuda_dev, K.flps_model_corr, FAG, obs, params, n, lag, 1, seed=710 + r)
        assert int(out["diag"][0, 2]) == 0 and int(out["diag"][0, 6]) == 5
        grads.append(out["gradient"][0].cpu().numpy())
    _zsum("grid N 2^20 T %d lag %d" % (nobs, lag), np.array(grads), fo.fa_gradient_targets(obs, phi, sv, se, lag)["grad_sum"])


def test_fully_adapted_gradient_spreads_less_than_the_bootstrap_one(cuda_dev):
    """Set 0 (phi 0.8, sigma_v 0.5, sigma_e 0.3), N = 4096, T = 60, lag 10, 16 replicates, the same u's (model 4 uses the
    first T - 1 time steps): the summed gradient's spread of model 4 is below 0.7 times model 1's for each parameter.
    The CPU restatement measured 0.37 / 0.29 / 0.42 for this set (sets 1, 2, 3: up to 0.73, 0.34, 0.17)."""
    from pmmh_qn_b200 import kernels as K
    n, nobs, lag, k, pset = 4096, 60, 10, 16, 0
    params = gi.LG_PARAM_SETS[pset]
    obs = _obs(nobs, pset)
    s = [np.asarray(_run(cuda_dev, K.flps_model_corr, m, obs, params, n, lag, k, seed=808)["gradient"].cpu().numpy())
         [:, :3].sum(axis=2).std(axis=0, ddof=1) for m in (LG, FAG)]
    print("spread model 1 %s model 4 %s ratio %s" % (np.round(s[0], 3), np.round(s[1], 3), np.round(s[1] / s[0], 3)))
    assert np.all(s[1] < 0.7 * s[0]), s


class ToyLGSSModel(object):
    """The attributes the estimators and CorrelatedPMMH read (the reference's model objects' interface)."""
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
        self.using_hessians = False

    def get_all_params(self):
        return np.array([self.params[k] for k in self.params])

    def check_parameters(self):
        p = self.params
        return abs(p['phi']) < 1.0 and p['sigma_v'] > 0.0 and p['sigma_e'] > 0.0

    def log_prior_gradient(self):
        return {k: 0.0 for k in self.params}

    def log_prior_hessian(self):
        return {k: 0.0 for k in self.params}


@pytest.mark.parametrize("fully_adapted", [True, False])
def test_estimator_equals_the_entry(cuda_dev, fully_adapted):
    import torch
    from pmmh_qn_b200 import DeviceRVS, LinearGaussianParticleMethodsCUDA
    from pmmh_qn_b200 import kernels as K
    n, nobs, lag = 1000, 50, 6
    params = gi.LG_PARAM_SETS[0]
    obs = _obs(nobs, 0)
    model = ToyLGSSModel(obs, params)
    est = LinearGaussianParticleMethodsCUDA(model, n, fixed_lag=lag, fully_adapted=fully_adapted)
    o = obs[1:] if fully_adapted else obs
    assert est.dim_rvs == (len(o), n + 1)
    rvs = gi.sv_rvs(n, len(o), 31)
    rvr, rvp = gi.split_particle(rvs, len(o))
    u = torch.from_numpy(np.ascontiguousarray(rvp.reshape(n, len(o)).T)).to(cuda_dev)
    par = torch.from_numpy(np.array([params], dtype=np.float64)).to(cuda_dev)
    ref = K.flps_model_corr(FAG if fully_adapted else LG, torch.from_numpy(np.ascontiguousarray(o)).to(cuda_dev), par,
                            torch.from_numpy(rvr).to(cuda_dev), u, lag=lag)
    extra = gp.log_p_y1(obs, params[1], params[2]) if fully_adapted else 0.0
    g = ref["gradient"][0].cpu().numpy()[:3].sum(axis=1)
    # host rvs: the entry's inputs bit for bit; a DeviceRVS takes Phi of r on the device (last-bit differences)
    for handle, tol in ((rvs, 0.0), (DeviceRVS.from_numpy_particle(rvs, cuda_dev), 1e-12)):
        assert est.smoother(model, rvs={'rvs': handle})
        r = est.results
        assert abs(r['log_like'] - (float(ref["log_like"][0]) + extra)) <= 1e-12 * abs(r['log_like'])
        for key, want in (('filt_state_est', ref["filt"][0]), ('smo_state_est', ref["smo"][0]),
                          ('state_trajectory', ref["traj"][0])):
            want = want.cpu().numpy()
            assert np.max(np.abs(r[key] - want)) <= tol * np.max(np.abs(want)), key
        for key in ('log_joint_gradient_estimate', 'gradient_internal'):
            assert np.max(np.abs(r[key] - g)) <= tol * np.max(np.abs(g)), key
        assert est.filter(model, rvs={'rvs': handle})
        assert abs(est.results['log_like'] - (float(ref["log_like"][0]) + extra)) <= 1e-12 * abs(r['log_like'])
    model.using_hessians = True
    assert not est.smoother(model, rvs={'rvs': rvs})


def test_correlated_pmmh_with_the_fully_adapted_estimator(cuda_dev):
    """100 iterations of CorrelatedPMMH (Langevin drift from the gradient) with device-resident correlated u."""
    from pmmh_qn_b200 import CorrelatedRVSState, LinearGaussianParticleMethodsCUDA
    from pmmh_qn_b200.parameter.cpmh import CorrelatedPMMH
    n, nobs = 500, 101
    params = gi.LG_PARAM_SETS[0]
    model = ToyLGSSModel(_obs(nobs, 0), params)
    est = LinearGaussianParticleMethodsCUDA(model, n, fixed_lag=10)
    st = CorrelatedRVSState.randn_particle(est.dim_rvs[0], n, cuda_dev, 0.3, seed=5)
    np.random.seed(11)
    sampler = CorrelatedPMMH(model, {'no_iters': 100, 'initial_params': params[:3], 'step_size': 0.03,
                                     'precond': (0.5, 0.5, 0.5), 'drift': True, 'rvs': st})
    sampler.run(est)
    h = sampler.state_history
    ll = np.array([h[i]['log_like'] for i in range(len(h))])
    acc = np.array([h[i]['accepted'] for i in range(1, len(h))])
    print("CPMH: acceptance %.2f, log-likelihood %.2f .. %.2f" % (acc.mean(), ll.min(), ll.max()))
    assert len(h) == 100 and np.all(np.isfinite(ll))
    assert 0.0 < acc.mean() < 1.0
