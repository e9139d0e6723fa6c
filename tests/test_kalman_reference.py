"""The exact fixed-lag Kalman reference (oracle/kalman.py) checks itself, and pins the NumPy restatement of the
linear Gaussian smoothers (oracle/generic_pf.py, models 1 and 2) to it: `filt`, `smo` and the gradient, per slot and
summed.  The targets are the exact conditional expectations the estimators' weights imply, so the comparisons carry no
lag-truncation allowance: a wrong observation index, a wrong weight generation, a double-counted or missing pair or an
off-by-one in the lag shows up as a bias.  CPU only."""
import numpy as np
import pytest

import generic_pf as gp
import golden_inputs as gi
import kalman as km

N, NOBS, SEEDS = 20000, 40, tuple(range(300, 312))
T_Q = 5.5           # |t| with 11 degrees of freedom (len(SEEDS) - 1) exceeds it with probability 2e-4: 36 summed checks
Z_MAX = 6.5         # per slot; z of 12 replicates is t-distributed with 11 degrees of freedom


def _fd_grad(obs, phi, sv, se, h=1e-6):
    p0 = np.array([phi, sv, se])
    out = np.zeros(3)
    for k in range(3):
        hi, lo = p0.copy(), p0.copy()
        hi[k] += h
        lo[k] -= h
        out[k] = (gp.kalman_loglike(obs, *hi) - gp.kalman_loglike(obs, *lo)) / (2.0 * h)
    return out


def _dense_moments(obs, phi, sv, se, c):
    """Mean and covariance of x_{0..T-1} given y_{1:c} by conditioning the joint Gaussian with numpy.linalg."""
    T = len(obs)
    idx = np.arange(1, T)
    # Cov(x_s, x_t) = sv^2 sum_{k=1}^{min(s,t)} phi^(s-k) phi^(t-k), x_0 = 0
    sxx = np.zeros((T, T))
    for s in idx:
        for t in idx:
            k = np.arange(1, min(s, t) + 1)
            sxx[s, t] = sv * sv * np.sum(phi ** (s - k) * phi ** (t - k))
    yo = np.arange(1, c + 1)
    syy = sxx[np.ix_(yo, yo)] + se * se * np.eye(c)
    sxy = sxx[:, yo]
    gain = np.linalg.solve(syy, sxy.T).T
    return gain @ np.asarray(obs)[yo], sxx - gain @ sxy.T


@pytest.mark.parametrize("pset", range(4))
def test_reference_with_full_lag_is_the_rts_smoother_and_its_score_the_likelihood_gradient(pset):
    phi, sv, se = gi.LG_PARAM_SETS[pset][:3]
    obs = gi.lg_obs(120, gi.LG_PARAM_SETS[pset])
    T = len(obs)
    tg = km.fixed_lag_targets(obs, phi, sv, se, lag=T)
    ms, _, _ = km.rts(km.kalman_filter(obs, phi, sv, se), T - 1, 0, phi)
    assert np.max(np.abs(tg["smo"] - ms)) <= 1e-12 * max(1.0, np.max(np.abs(ms)))
    fd = _fd_grad(obs, phi, sv, se)
    assert np.all(np.abs(tg["grad_sum"] - fd) <= 1e-7 * np.maximum(np.abs(fd), 1.0)), (tg["grad_sum"], fd)
    assert tg["grad"][:, 0].tolist() == [0.0, 0.0, 0.0]
    # model 2's tail conditions on everything the series holds, as model 1's does
    fa = km.fixed_lag_targets(obs, phi, sv, se, lag=T, fully_adapted=True)
    assert np.max(np.abs(fa["smo"] - ms[:T - 1])) <= 1e-12 * max(1.0, np.max(np.abs(ms)))


@pytest.mark.parametrize("pset", range(4))
@pytest.mark.parametrize("lag", [2, 3, 5])
def test_reference_against_dense_conditioning(pset, lag):
    """T = 8: every mean, second moment and score target against dense Gaussian conditioning (no recursion shared)."""
    phi, sv, se = gi.LG_PARAM_SETS[pset][:3]
    obs = gi.lg_obs(8, gi.LG_PARAM_SETS[pset], seed=99)
    T = len(obs)
    for fa in (False, True):
        tg = km.fixed_lag_targets(obs, phi, sv, se, lag, fully_adapted=fa)
        n = T - 1 if fa else T
        for t in range(n):
            c = min(t + lag - 1, n - 1) + (1 if fa else 0)
            mean, cov = _dense_moments(obs, phi, sv, se, c)
            assert abs(tg["smo"][t] - mean[t]) <= 1e-12, (fa, t)
        if fa:
            continue
        assert len(tg["mom"]) == T - 1
        for t, (c, m0, p0, m1, p1, c01) in enumerate(tg["mom"]):
            mean, cov = _dense_moments(obs, phi, sv, se, c)
            e00, e11, e01 = cov[t, t] + mean[t] ** 2, cov[t + 1, t + 1] + mean[t + 1] ** 2, cov[t, t + 1] + mean[t] * mean[t + 1]
            assert abs(p0 + m0 * m0 - e00) <= 1e-12 and abs(p1 + m1 * m1 - e11) <= 1e-12
            assert abs(c01 + m0 * m1 - e01) <= 1e-12
            g = np.array([(e01 - phi * e00) / sv ** 2,
                          ((e11 - 2 * phi * e01 + phi * phi * e00) / sv ** 2 - 1.0) / sv,
                          (((obs[t + 1] - mean[t + 1]) ** 2 + cov[t + 1, t + 1]) / se ** 2 - 1.0) / se])
            assert np.all(np.abs(tg["grad"][:, t + 1] - g) <= 1e-12 * np.maximum(np.abs(g), 1.0)), (t, tg["grad"][:, t + 1], g)
    # filt targets: model 1 E[x_t | y_1:t], model 2 E[x_t | y_1:t+1]
    f1, f2 = km.filtered_means(obs, phi, sv, se), km.fa_filtered_means(obs, phi, sv, se)
    for t in range(1, T):
        assert abs(f1[t] - _dense_moments(obs, phi, sv, se, t)[0][t]) <= 1e-12
        if t < T - 1:
            assert abs(f2[t] - _dense_moments(obs, phi, sv, se, t + 1)[0][t]) <= 1e-12


def _zcheck(name, reps, exact, skip_zero_slots=False):
    """Per slot z = (mean - exact) / (s / sqrt(K)) with s floored at its median over the slots (a handful of replicates
    estimates s poorly): RMS of z <= 1.5, largest |z| <= Z_MAX."""
    reps = np.asarray(reps)
    k = reps.shape[0]
    mean, s = reps.mean(axis=0), reps.std(axis=0, ddof=1)
    live = s > 0 if skip_zero_slots else np.ones_like(s, dtype=bool)
    s = np.maximum(s, np.median(s[live]))
    z = (mean - exact)[live] / (s[live] / np.sqrt(k))
    rms, zmax = float(np.sqrt(np.mean(z * z))), float(np.max(np.abs(z)))
    assert rms <= 1.5 and zmax <= Z_MAX, "%s: RMS z %.2f, max |z| %.2f at slot %d" % (
        name, rms, zmax, int(np.flatnonzero(live)[np.argmax(np.abs(z))]))
    return rms, zmax


def _runs(model, obs, n):
    out = []
    for seed in SEEDS:
        rvr, rvp = gi.split_particle(gi.sv_rvs(n, len(obs), seed), len(obs))
        out.append([gp.flps_generic(model, obs, rvr, rvp, n, lag) for lag in (2, 4, 10)])
    return out


@pytest.mark.parametrize("pset", range(4))
def test_linear_gaussian_restatement_against_exact_fixed_lag_targets(pset):
    """Model 1 (bootstrap filter): filt, smo per slot, gradient per slot and summed."""
    params = gi.LG_PARAM_SETS[pset]
    phi, sv, se = params[:3]
    obs = gi.lg_obs(NOBS, params, seed=4711 + pset)
    runs = _runs(gp.LinearGaussian(params), obs, N)
    _zcheck("filt", [r[0]["filt"][1:] for r in runs], km.filtered_means(obs, phi, sv, se)[1:])
    for li, lag in enumerate((2, 4, 10)):
        tg = km.fixed_lag_targets(obs, phi, sv, se, lag)
        _zcheck("lag %d smo" % lag, [r[li]["smo"][1:] for r in runs], tg["smo"][1:])
        g = np.array([r[li]["gradient"] for r in runs])
        assert np.all(g[:, :, 0] == 0.0) and np.all(g[:, 3] == 0.0)
        for q, pname in enumerate(("phi", "sigma_v", "sigma_e")):
            _zcheck("lag %d gradient %s" % (lag, pname), g[:, q, 1:], tg["grad"][q, 1:])
            tot = g[:, q].sum(axis=1)
            err, se_m = tot.mean() - tg["grad_sum"][q], tot.std(ddof=1) / np.sqrt(len(tot))
            assert abs(err) <= T_Q * se_m, "lag %d summed gradient %s: %.4g vs exact %.4g (%.1f se)" % (
                lag, pname, tot.mean(), tg["grad_sum"][q], err / se_m)


@pytest.mark.parametrize("pset", range(4))
def test_fully_adapted_restatement_against_exact_fixed_lag_targets(pset):
    """Model 2 (fully adapted filter, run on obs[1:]): filt = E[x_t | y_1:t+1], smo per slot, gradient rows 0."""
    params = gi.LG_PARAM_SETS[pset]
    phi, sv, se = params[:3]
    obs = gi.lg_obs(NOBS, params, seed=4711 + pset)
    runs = _runs(gp.LinearGaussianFullyAdapted(params), obs[1:], N // 4)
    _zcheck("filt", [r[0]["filt"][1:] for r in runs], km.fa_filtered_means(obs, phi, sv, se)[1:])
    for li, lag in enumerate((2, 4, 10)):
        tg = km.fixed_lag_targets(obs, phi, sv, se, lag, fully_adapted=True)
        _zcheck("lag %d smo" % lag, [r[li]["smo"][1:] for r in runs], tg["smo"][1:])
        assert all(np.all(r[li]["gradient"] == 0.0) for r in runs)
