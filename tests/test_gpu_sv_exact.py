"""Model id 8 (the SV model with the exact fixed-lag score and a Hessian, csrc/pf_model.cuh SvLeverageExact):

- against the restatement (tests/sv_exact_oracle.py) on the chain kernel, the one-problem grid kernel and a team batch,
  lag 2 and 10: ancestors exact, log_like 1e-10 relative, gradient per slot 1e-9 and hess1 / hess2 1e-10 of their
  largest entry (replayed on the kernel's own history);
- bit-identity with model 0: filt, log_like, traj, diag and the history on the chain kernel, and the filter entries on
  both kernels; a team batch bit-identical to its one-problem runs, the Hessian included;
- the restatement in the shape of the quadrature comparison (waves of teams, the Hessian, no history);
- against the quadrature oracle (tests/sv_quadrature.py) over replicates: per-slot and summed gradient, smoothed means,
  the summed hess1 and hess2;
- the estimators with pairing='exact' publish what the entries return, and the gradient-driven correlated PMMH sampler
  runs on them unchanged."""
import numpy as np
import pytest

import generic_pf as gp
import golden_inputs as gi
import sv_exact_oracle as so
import sv_quadrature as sq
from helpers import to_time_major
from toy_models import ToySVModel

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_KERNEL = 2, 6
CHAIN, GRID = 3, 5
SV, SVX = 0, 8


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def _np(out, b=None):
    return {k: (v.cpu().numpy() if b is None else v[b].cpu().numpy()) for k, v in out.items() if not k.startswith("_")}


def _inputs(cuda_dev, n, nobs, pset, seed, batch=1):
    """host (obs, params, rvr [B][nobs], rvp [B][nobs * n]) and the device inputs"""
    obs = gi.sv_obs(nobs, gi.SV_PARAM_SETS[0], seed=seed)
    params = np.array(gi.SV_PARAM_SETS[pset], dtype=np.float64)
    rv = [gi.split_particle(gi.sv_rvs(n, nobs, seed + b), nobs) for b in range(batch)]
    rvr = np.array([r[0] for r in rv])
    rvp = np.array([r[1] for r in rv])
    u = np.array([to_time_major(r[1], n, nobs) for r in rv])
    d = _dev(cuda_dev, obs, np.tile(params, (batch, 1)), rvr, u)
    return (obs, params, rvr, rvp), d


def _weights(params, obs, X):
    m = gp.SvLeverage(params)
    W = np.zeros_like(X)
    W[0] = 1.0 / X.shape[1]
    for i in range(1, X.shape[0]):
        lw = m.logw(X[i], obs[i])
        sh = np.exp(lw - np.max(lw))
        W[i] = sh / np.sum(sh)
    return W


def _check_vs_restatement(res, host, n, lag, hess):
    obs, params, rvr, rvp = host
    ref = so.flps_sv_exact(params, obs, rvr, rvp, n, lag, dumps=True)
    assert np.array_equal(res["A"], ref["A"])
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"])
    X, A = res["X"], res["A"].astype(np.int64)
    r = so.predictive_replay(so.SvLeverageExact(params), obs, X, A, _weights(params, obs, X), lag, hessian=hess)
    g = r[0] if hess else r
    assert np.max(np.abs(res["gradient"] - g)) <= 1e-9 * np.max(np.abs(g)), (res["gradient"] - g)
    assert np.all(res["gradient"][:, -1] == 0.0)
    if hess:
        for got, want in ((res["hess1"], r[1]), (res["hess2"], r[2])):
            assert np.max(np.abs(got - want)) <= 1e-10 * np.max(np.abs(want)), (got, want)


@pytest.mark.parametrize("lag", [2, 10])
@pytest.mark.parametrize("pset", [0, 2])
def test_against_restatement_on_every_kernel(cuda_dev, pset, lag):
    from pmmh_qn_b200 import kernels as K
    nobs = 40
    for n in (1000, 8192):       # chain kernel, one-problem grid kernel
        host, (obs_d, par, rvr, u) = _inputs(cuda_dev, n, nobs, pset, 11 * lag + pset)
        res = _np(K.flps_model_corr(SVX, obs_d, par, rvr, u, lag=lag, store_history=True), 0)
        assert int(res["diag"][DIAG_KERNEL]) == (CHAIN if n <= 4096 else GRID)
        assert int(res["diag"][DIAG_STATUS]) == 0
        _check_vs_restatement(res, (host[0], host[1], host[2][0], host[3][0]), n, lag, False)
    n, B = 8192, 2              # team batch with the Hessian
    host, (obs_d, par, rvr, u) = _inputs(cuda_dev, n, nobs, pset, 500 + lag, batch=B)
    out = K.flps_model_batch_corr(SVX, obs_d, par, rvr, u, lag=lag, compute_hessian=1, store_history=True)
    for b in range(B):
        res = _np(out, b)
        assert int(res["diag"][DIAG_KERNEL]) == GRID and int(res["diag"][DIAG_STATUS]) == 0
        _check_vs_restatement(res, (host[0], host[1], host[2][b], host[3][b]), n, lag, True)


@pytest.mark.parametrize("n,batch", [(1000, 3), (1 << 14, 1)])
def test_bit_identical_to_model_0(cuda_dev, n, batch):
    """the smoother on the chain kernel (which runs every model through the same code) and the filter entries on both
    kernels; the grid kernel runs model 0 on its SV path and model 8 on the generic one, so there the smoother's
    log-likelihood agrees to rounding"""
    from pmmh_qn_b200 import kernels as K
    _, (obs_d, par, rvr, u) = _inputs(cuda_dev, n, 60, 1, 77, batch=batch)
    m0, m8 = (_np(K.flps_model_corr(m, obs_d, par, rvr, u, lag=10, store_history=True)) for m in (SV, SVX))
    if n <= 4096:
        for k in ("filt", "log_like", "traj", "diag", "X", "A"):
            assert np.array_equal(m0[k], m8[k]), k
    else:
        assert np.all(np.abs(m0["log_like"] - m8["log_like"]) <= 1e-12 * np.abs(m0["log_like"]))
    assert not np.array_equal(m0["gradient"], m8["gradient"])
    f0, f8 = (_np(K.filter_model_corr(m, obs_d, par, rvr, u, store_history=True)) for m in (SV, SVX))
    for k in ("filt", "log_like", "traj", "diag", "X", "A"):
        assert np.array_equal(f0[k], f8[k]), k


def test_team_batch_bit_identical_to_one_problem_runs(cuda_dev):
    from pmmh_qn_b200 import kernels as K
    n, B = 1 << 14, 6
    _, (obs_d, par, rvr, u) = _inputs(cuda_dev, n, 40, 0, 900, batch=B)
    import torch
    par = par + 0.01 * (torch.arange(B, dtype=torch.float64, device=cuda_dev) % 3)[:, None]
    bt = _np(K.flps_model_batch_corr(SVX, obs_d, par, rvr, u, lag=10, compute_hessian=1))
    assert np.all(bt["diag"][:, DIAG_STATUS] == 0)
    for b in range(B):
        one = _np(K.flps_model_batch_corr(SVX, obs_d, par[b:b + 1], rvr[b:b + 1], u[b:b + 1], lag=10, compute_hessian=1), 0)
        for k in ("filt", "smo", "log_like", "gradient", "traj", "diag", "hess1", "hess2"):
            assert np.array_equal(bt[k][b], one[k]), (b, k)
    # without the Hessian, the batch entry gives the one-problem entry's outputs
    one = _np(K.flps_model_corr(SVX, obs_d, par[:1], rvr[:1], u[:1], lag=10), 0)
    b0 = _np(K.flps_model_batch_corr(SVX, obs_d, par[:1], rvr[:1], u[:1], lag=10), 0)
    for k in ("filt", "smo", "log_like", "gradient", "traj"):
        assert np.array_equal(b0[k], one[k]), k


def _z(reps, exact):
    s = reps.std(axis=0, ddof=1)
    live = s > 0.0
    return (reps.mean(axis=0) - exact)[live] / (s[live] / np.sqrt(reps.shape[0])), live


def _quad_inputs(cuda_dev, k, seed):
    """the replicates of the quadrature comparisons: obs (host), and obs, params, rvr, u on the device"""
    import torch
    params = gi.SV_PARAM_SETS[0]
    nobs, n = 20, 1 << 14
    obs = gi.sv_obs(nobs, params, seed=2025)
    g = torch.Generator(device=cuda_dev)
    g.manual_seed(seed)
    u = torch.randn((k, nobs, n), dtype=torch.float64, device=cuda_dev, generator=g)
    rvr = torch.rand((k, nobs), dtype=torch.float64, device=cuda_dev, generator=g)
    par = torch.from_numpy(np.tile(np.asarray(params, dtype=np.float64), (k, 1))).to(cuda_dev)
    return obs, _dev(cuda_dev, obs)[0], par, rvr, u


def test_restatement_in_the_quadrature_shape(cuda_dev):
    """the quadrature comparison's own shape -- 64 problems of N = 2^14 in waves of teams (8 CTAs each), the Hessian, no
    history -- against the restatement run on the same u and resampling uniforms: log_like 1e-10 relative (which the
    same ancestors give), gradient 1e-9, hess1 / hess2 1e-10 of their largest entry, every problem"""
    from pmmh_qn_b200 import kernels as K
    k, lag = 64, 10
    obs, obs_d, par, rvr, u = _quad_inputs(cuda_dev, k, 7)
    out = _np(K.flps_model_batch_corr(SVX, obs_d, par, rvr, u, lag=lag, compute_hessian=1))
    assert np.all(out["diag"][:, DIAG_STATUS] == 0) and np.all(out["diag"][:, DIAG_KERNEL] == GRID)
    rvr_h, u_h, n = rvr.cpu().numpy(), u.cpu().numpy(), u.shape[2]
    for b in range(k):
        ref = so.flps_sv_exact(gi.SV_PARAM_SETS[0], obs, rvr_h[b], np.ascontiguousarray(u_h[b].T).ravel(), n, lag,
                               hessian=True)
        assert abs(float(out["log_like"][b]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"]), b
        assert np.max(np.abs(out["gradient"][b] - ref["gradient"])) <= 1e-9 * np.max(np.abs(ref["gradient"])), b
        for kk in ("hess1", "hess2"):
            assert np.max(np.abs(out[kk][b] - ref[kk])) <= 1e-10 * np.max(np.abs(ref[kk])), (b, kk)


@pytest.mark.parametrize("seed", [7, 8])
def test_against_quadrature(cuda_dev, seed):
    """n_obs = 20, lag 10, N = 2^14, 128 replicates in one team batch at the data-generating values (rho = -0.5),
    against the exact fixed-lag targets of tests/sv_quadrature.py, |z| <= 5 per entry: the per-slot gradient and its sum
    over the slots, the smoothed means, and the summed hess1 and hess2 (which pin hess1 + hess2 - g g'); model 0's
    summed gradient on the same replicates is reported beside"""
    from pmmh_qn_b200 import kernels as K
    params = gi.SV_PARAM_SETS[0]
    k, lag = 128, 10
    obs, obs_d, par, rvr, u = _quad_inputs(cuda_dev, k, seed)
    out = _np(K.flps_model_batch_corr(SVX, obs_d, par, rvr, u, lag=lag, compute_hessian=1))
    assert np.all(out["diag"][:, DIAG_STATUS] == 0)
    m = so.SvLeverageExact(params)
    q = sq.quadrature_targets(m, m.trans_sd(), obs, lag, params[0] - 8.0, params[0] + 8.0, m=601, pair_y=0,
                              hessian=True)
    m0 = _np(K.flps_model_batch_corr(SV, obs_d, par, rvr, u, lag=lag))
    for name, gr in (("model 8", out["gradient"]), ("model 0", m0["gradient"])):
        z, _ = _z(gr.sum(axis=2), q["score"].sum(axis=1))
        print(name, "summed gradient", np.round(gr.sum(axis=2).mean(axis=0), 4).tolist(), "exact",
              np.round(q["score"].sum(axis=1), 4).tolist(), "z", np.round(z, 2).tolist())
    cases = (("gradient", out["gradient"], q["score"]), ("summed gradient", out["gradient"].sum(axis=2),
             q["score"].sum(axis=1)), ("smo", out["smo"][:, 1:], q["smo"][1:]),
             ("hess1", out["hess1"], q["hess1"].sum(axis=0)), ("hess2", out["hess2"], q["hess2"].sum(axis=0)))
    for name, reps, exact in cases:
        z, _ = _z(reps, exact)
        print(name, "max |z|", np.round(np.max(np.abs(z)), 2))
    for name, reps, exact in cases:
        z, _ = _z(reps, exact)
        assert np.all(np.abs(z) <= 5.0), (name, z)


@pytest.mark.parametrize("hess", [False, True])
def test_estimator_publishes_the_entrys_outputs(cuda_dev, hess):
    from pmmh_qn_b200 import ParticleMethodsCUDA
    from pmmh_qn_b200 import kernels as K
    n, nobs, lag = 1000, 120, 10
    model = ToySVModel(gi.sv_obs(nobs), gi.SV_PARAM_SETS[0])
    model.using_hessians = hess
    rvs = gi.sv_rvs(n, nobs, 31)
    rvr, rvp = gi.split_particle(rvs, nobs)
    obs_d, par, rvr_d, u = _dev(cuda_dev, gi.sv_obs(nobs), np.array([gi.SV_PARAM_SETS[0]]), rvr[None],
                                to_time_major(rvp, n, nobs)[None])
    if hess:
        ref = _np(K.flps_model_batch_corr(SVX, obs_d, par, rvr_d, u, lag=lag, compute_hessian=1), 0)
    else:
        ref = _np(K.flps_model_corr(SVX, obs_d, par, rvr_d, u, lag=lag), 0)
    est = ParticleMethodsCUDA(model, n, fixed_lag=lag, pairing='exact')
    assert est.settings['pairing'] == 'exact'
    assert est.smoother(model, rvs={'rvs': rvs})
    r = est.results
    assert r['log_like'] == float(ref["log_like"])
    assert np.array_equal(r['smo_state_est'], ref["smo"]) and np.array_equal(r['filt_state_est'], ref["filt"])
    g = np.nansum(ref["gradient"], axis=1)
    assert np.array_equal(r['log_joint_gradient_estimate'], g)
    if hess:
        assert np.array_equal(r['log_joint_hessian_estimate'], ref["hess1"] + ref["hess2"] - np.outer(g, g))
    # the reference pairing is unchanged by the option
    base = ParticleMethodsCUDA(model, n, fixed_lag=lag)
    assert base.settings['pairing'] == 'reference' and base.smoother(model, rvs={'rvs': rvs})
    assert not np.array_equal(base.results['log_joint_gradient_estimate'], g)


def test_estimator_refuses_sizes_the_entries_refuse(cuda_dev):
    from pmmh_qn_b200 import ParticleMethodsCUDA
    from pmmh_qn_b200._lib import PmmhError
    model = ToySVModel(gi.sv_obs(8), gi.SV_PARAM_SETS[0])
    with pytest.raises(PmmhError):
        ParticleMethodsCUDA(model, 1000, fixed_lag=10, pairing='exact')     # n_obs < lag + 1
    model = ToySVModel(gi.sv_obs(200), gi.SV_PARAM_SETS[0])
    with pytest.raises(PmmhError):
        ParticleMethodsCUDA(model, 1000, fixed_lag=11, pairing='exact')     # lag > 10
    with pytest.raises(ValueError):
        ParticleMethodsCUDA(model, 1000, pairing='other')


@pytest.mark.parametrize("n,hess", [(1000, False), (1000, True), (8192, False)])
def test_batched_backend_exact(cuda_dev, n, hess):
    from pmmh_qn_b200 import ParticleMethodsCUDA
    from pmmh_qn_b200.parameter.lockstep import _Request
    from pmmh_qn_b200.state.particle_methods.batched import BatchedParticleMethodsCUDA
    nobs, B = 60, 3
    models = [ToySVModel(gi.sv_obs(nobs), np.array(gi.SV_PARAM_SETS[0]) + 0.01 * b) for b in range(B)]
    for m in models:
        m.using_hessians = hess
    backend = BatchedParticleMethodsCUDA(models[0], no_particles=n, pairing='exact')
    one = ParticleMethodsCUDA(models[0], no_particles=n, pairing='exact')
    rvs = [gi.sv_rvs(n, nobs, 40 + b) for b in range(B)]
    reqs = [_Request(b, "smoother", models[b], {'rvs': {'rvs': rvs[b]}}, dict(backend.settings)) for b in range(B)]
    backend.evaluate_batch(reqs)
    for b in range(B):
        assert reqs[b].ok
        assert one.smoother(models[b], rvs={'rvs': rvs[b]})
        for k in ('log_like', 'gradient_internal') + (('hessian_internal',) if hess else ()):
            assert np.array_equal(reqs[b].results[k], one.results[k]), k


def test_gradient_sampler_drives_the_exact_pairing(cuda_dev):
    """the correlated PMMH sampler with Langevin drift (parameter/cpmh.py, the reference's sampler interface) runs
    ParticleMethodsCUDA(pairing='exact') unchanged, alone and through the lock-step batched backend (chains bit-identical
    either way); its proposals follow model 8's gradient, so the trace differs from the reference pairing's"""
    from pmmh_qn_b200 import ParticleMethodsCUDA
    from pmmh_qn_b200.parameter.lockstep import LockstepRunner
    from pmmh_qn_b200.state.particle_methods.batched import BatchedParticleMethodsCUDA
    from test_gpu_lockstep import _sampler, _trace
    n, nobs, B = 500, 61, 3
    seeds = [300 + k for k in range(B)]
    solo = {}
    for pairing in ("exact", "reference"):
        solo[pairing] = []
        for k in range(B):
            s = _sampler(nobs, k)
            np.random.seed(seeds[k])
            s.run(ParticleMethodsCUDA(s.model, no_particles=n, pairing=pairing))
            solo[pairing].append(_trace(s))
    chains = [_sampler(nobs, k) for k in range(B)]
    backend = BatchedParticleMethodsCUDA(chains[0].model, no_particles=n, pairing='exact')
    LockstepRunner(chains, backend, seeds=seeds).run()
    for k in range(B):
        params, ll, acc = solo["exact"][k]
        assert np.all(np.isfinite(params)) and np.all(np.isfinite(ll))
        for a, b in zip(_trace(chains[k]), solo["exact"][k]):
            assert np.array_equal(a, b), k
    assert any(t[2][1:].sum() > 0 for t in solo["exact"])
    assert any(not np.array_equal(a[0], b[0]) for a, b in zip(solo["exact"], solo["reference"]))
