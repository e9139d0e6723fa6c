"""The Hessian of the fully adapted linear Gaussian filter (model id 6, csrc/pf_model.cuh: model 4 with the generic
Hessian branch).  CPU only:

- the hooks (score_main / score_last and hess_main / hess_last) against central differences of the log densities;
- the exact per-slot hess1 targets (tests/fa_hessian_oracle.py hess1_targets) against dense Gaussian conditioning, and
  the restatement's hess1 against them at large N;
- the restatement's hess1 + hess2 - g g' against the exact Hessian of the Kalman log-likelihood (n' = 20, lag 10,
  phi = 0.5: lag truncation is negligible), within the spread of independent replicates;
- three one-line mispairings of alpha (tests/fa_hessian_oracle.py) fail that comparison.
"""
import numpy as np
import pytest

import fa_hessian_oracle as fh
import generic_pf as gp
import golden_inputs as gi
from test_fa_gradient_reference import _dense_moments

PARAMS = (0.5, 0.6, 0.4, 0.0)      # phi ~ 0.5: the lag-10 truncation is below the replicate spread
NPRIME, LAG, N, SEEDS = 20, 10, 2000, tuple(range(40))
Z = 5.0                            # |mean - exact| <= Z s / sqrt(K) per entry


def _logdens_main(p, curr, nxt, y):
    phi, sv, se = p
    r, ry = nxt - phi * curr, y - nxt
    return -np.log(sv) - 0.5 * r * r / (sv * sv) - np.log(se) - 0.5 * ry * ry / (se * se)


def _logdens_last(p, x, y):
    phi, sv, se = p
    s2 = sv * sv + se * se
    r = y - phi * x
    return -0.5 * np.log(s2) - 0.5 * r * r / s2


def _fd(f, p0, h=1e-5):
    """gradient and Hessian of f at p0 by central differences"""
    g, hs = np.zeros(3), np.zeros((3, 3))
    for a in range(3):
        ea = np.eye(3)[a] * h
        g[a] = (f(p0 + ea) - f(p0 - ea)) / (2 * h)
        for b in range(3):
            eb = np.eye(3)[b] * h
            hs[a, b] = (f(p0 + ea + eb) - f(p0 + ea - eb) - f(p0 - ea + eb) + f(p0 - ea - eb)) / (4 * h * h)
    return g, hs


@pytest.mark.parametrize("pset", range(4))
def test_hooks_against_finite_differences(pset):
    params = gi.LG_PARAM_SETS[pset]
    m = fh.LinearGaussianFullyAdaptedHess(params)
    p0 = np.array(params[:3], dtype=np.float64)
    rng = np.random.default_rng(pset)
    for curr, nxt, y in rng.normal(size=(5, 3)):
        g, hs = _fd(lambda p: _logdens_main(p, curr, nxt, y), p0)
        assert np.max(np.abs(m.score_main(curr, nxt, y)[:3] - g)) <= 1e-6 * max(np.max(np.abs(g)), 1.0)
        assert np.max(np.abs(m.hess_main(curr, nxt, y)[:3, :3] - hs)) <= 1e-6 * max(np.max(np.abs(hs)), 1.0)
        g, hs = _fd(lambda p: _logdens_last(p, curr, y), p0)
        assert np.max(np.abs(m.score_last(curr, y)[:3] - g)) <= 1e-6 * max(np.max(np.abs(g)), 1.0)
        assert np.max(np.abs(m.hess_last(curr, y)[:3, :3] - hs)) <= 1e-6 * max(np.max(np.abs(hs)), 1.0)
        assert np.all(m.hess_main(curr, nxt, y)[3] == 0.0) and np.all(m.hess_last(curr, y)[:, 3] == 0.0)


@pytest.mark.parametrize("pset", range(4))
@pytest.mark.parametrize("lag", [2, 3, 5])
def test_hess1_targets_against_dense_conditioning(pset, lag):
    """T = 8: every slot's E[H_k] from dense Gaussian conditioning (no recursion shared)."""
    phi, sv, se = gi.LG_PARAM_SETS[pset][:3]
    obs = gi.lg_obs(8, gi.LG_PARAM_SETS[pset], seed=99)
    T = len(obs)
    n = T - 1
    tg = fh.hess1_targets(obs, phi, sv, se, lag)
    for k in range(n - 1):
        mean, cov = _dense_moments(obs, phi, sv, se, min(k + lag - 1, n - 1) + 1)
        e00, e11 = cov[k, k] + mean[k] ** 2, cov[k + 1, k + 1] + mean[k + 1] ** 2
        e01 = cov[k, k + 1] + mean[k] * mean[k + 1]
        er2 = e11 - 2 * phi * e01 + phi * phi * e00
        ery2 = (obs[k + 1] - mean[k + 1]) ** 2 + cov[k + 1, k + 1]
        h = np.array([[-e00 / sv ** 2, -2 * (e01 - phi * e00) / sv ** 3, 0.0],
                      [-2 * (e01 - phi * e00) / sv ** 3, 1 / sv ** 2 - 3 * er2 / sv ** 4, 0.0],
                      [0.0, 0.0, 1 / se ** 2 - 3 * ery2 / se ** 4]])
        assert np.max(np.abs(tg[k] - h)) <= 1e-12 * max(np.max(np.abs(h)), 1.0), (k, tg[k], h)
    # last slot: E[hess_last(x_{T-2}, y_{T-1}) | y_{1:T-1}] by Gauss-Hermite quadrature of the hook
    mean, cov = _dense_moments(obs, phi, sv, se, T - 1)
    xs, ws = np.polynomial.hermite_e.hermegauss(12)
    x = mean[T - 2] + np.sqrt(cov[T - 2, T - 2]) * xs
    want = np.sum(fh.LinearGaussianFullyAdaptedHess(gi.LG_PARAM_SETS[pset]).hess_last(x, obs[T - 1])[:3, :3] * ws,
                  axis=2) / np.sqrt(2 * np.pi)
    assert np.max(np.abs(tg[n - 1] - want)) <= 1e-10 * max(np.max(np.abs(want)), 1.0)


@pytest.fixture(scope="module")
def replicates():
    """the restatement at N = 2000 on n' = 20, lag 10, over 40 independent u: {mutation: [K][3][3] estimates}, and the
    first run's hess1 / per-run outputs"""
    obs = gi.lg_obs(NPRIME + 1, PARAMS, seed=4242)
    out = {m: [] for m in (None, "alpha_own", "alpha_read", "drop_last")}
    h1 = []
    for seed in SEEDS:
        rvr, rvp = gi.split_particle(gi.sv_rvs(N, NPRIME, 700 + seed), NPRIME)
        base = fh.fo.flps_fa_grad(PARAMS, obs[1:], rvr, rvp, N, LAG, dumps=True)
        model = fh.LinearGaussianFullyAdaptedHess(PARAMS)
        for m in out:
            r = dict(base)
            r["hess1"], r["hess2"] = fh.predictive_hessian(model, obs[1:], base["X"], base["A"], base["W"], LAG, m)
            out[m].append(fh.hessian_estimate(r))
            if m is None:
                h1.append(r["hess1"][:3, :3])
    return obs, {m: np.array(v) for m, v in out.items()}, np.array(h1)


def _z(reps, exact):
    k = reps.shape[0]
    return (reps.mean(axis=0) - exact) / (reps.std(axis=0, ddof=1) / np.sqrt(k))


def test_restatement_hess1_against_exact_targets(replicates):
    obs, _, h1 = replicates
    exact = fh.hess1_targets(obs, *PARAMS[:3], LAG).sum(axis=0)
    z = _z(h1, exact)
    print("hess1 z", np.round(z, 2))
    assert np.all(np.abs(z[np.isfinite(z)]) <= Z), z


def test_restatement_hessian_against_the_kalman_hessian(replicates):
    obs, est, _ = replicates
    exact = fh.kalman_hessian(obs, *PARAMS[:3])
    z = _z(est[None], exact)
    print("exact", np.round(exact, 3), "mean", np.round(est[None].mean(axis=0), 3), "z", np.round(z, 2))
    assert np.all(np.abs(z) <= Z), z


@pytest.mark.parametrize("mutation", ["alpha_own", "alpha_read", "drop_last"])
def test_mispairings_are_rejected(replicates, mutation):
    obs, est, _ = replicates
    z = _z(est[mutation], fh.kalman_hessian(obs, *PARAMS[:3]))
    print(mutation, "max |z|", float(np.max(np.abs(z))))
    assert np.max(np.abs(z)) > Z, z


def test_kalman_hessian_matches_the_gradient_targets():
    """The central-difference Hessian is the derivative of generic_pf.kalman_loglike's score."""
    obs = gi.lg_obs(NPRIME + 1, PARAMS, seed=4242)
    h = fh.kalman_hessian(obs, *PARAMS[:3])
    d = 1e-5
    for a in range(3):
        e = np.eye(3)[a] * d
        gp_, gm = (fh.fo.fa_gradient_targets(obs, *(np.array(PARAMS[:3]) + s * e), lag=len(obs))["grad_sum"]
                   for s in (1.0, -1.0))
        assert np.max(np.abs((gp_ - gm) / (2 * d) - h[a])) <= 1e-5 * np.max(np.abs(h))
    assert np.isfinite(gp.kalman_loglike(obs, *PARAMS[:3]))
