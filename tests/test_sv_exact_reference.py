"""CPU checks of model id 8 (csrc/pf_model.cuh SvLeverageExact) and of its oracles:

- the hooks of the restatement (tests/sv_exact_oracle.py, the device hooks formula for formula) against central
  differences: score_main / score_first of the transition log-density in theta = (mu, atanh phi, log sigma_v, atanh rho),
  hess_main / hess_first of the scores;
- the quadrature oracle (tests/sv_quadrature.py) against oracle/kalman.py with the linear Gaussian callbacks, and against
  Fisher's and Louis' identities for the SV model at full smoothing (lag = n_obs: the score slots sum to the gradient of
  log_like, and hess1 + hess2 - g g' of its targets is the Hessian of log_like);
- predictive_replay against the existing restatements of models 4 and 6 on their own histories;
- the restatement's per-slot gradient against the quadrature targets over replicates, and model 0's restatement
  (the reference's pairing, Q5 / Q6) against the same targets at rho = -0.5, where its bias is resolved by far.
"""
import numpy as np
import pytest

import fa_gradient_oracle as fo
import fa_hessian_oracle as fh
import generic_pf as gp
import golden_inputs as gi
import kalman as km
import sv_exact_oracle as so
import sv_quadrature as sq

THETA = [np.array([p[0], np.arctanh(p[1]), np.log(p[2]), np.arctanh(p[3])]) for p in gi.SV_PARAM_SETS]


def _make(theta):
    m = so.SvLeverageExact.from_theta(theta)
    return m, m.trans_sd()


def _points(seed):
    rs = np.random.RandomState(seed)
    return rs.normal(size=7) * 0.8, rs.normal(size=7) * 0.8, rs.normal(size=7) * 1.5


def _diff(f, theta, h):
    e = np.eye(4) * h
    return np.array([(f(theta + e[a]) - f(theta - e[a])) / (2.0 * h) for a in range(4)])


@pytest.mark.parametrize("pset", [0, 1, 2])
def test_hooks_against_central_differences(pset):
    theta = THETA[pset]
    curr, nxt, y = _points(pset)
    curr, nxt = curr + theta[0], nxt + theta[0]
    m = so.SvLeverageExact.from_theta(theta)
    first_lp = lambda t: (lambda mm: mm.trans_logpdf(np.full_like(nxt, mm.mu), nxt, y))(so.SvLeverageExact.from_theta(t))
    cases = (
        ("score_main", m.score_main(curr, nxt, y),
         _diff(lambda t: so.SvLeverageExact.from_theta(t).trans_logpdf(curr, nxt, y), theta, 1e-6)),
        ("score_first", m.score_first(nxt, y), _diff(first_lp, theta, 1e-6)),
        ("hess_main", m.hess_main(curr, nxt, y),
         _diff(lambda t: so.SvLeverageExact.from_theta(t).score_main(curr, nxt, y), theta, 1e-5)),
        ("hess_first", m.hess_first(nxt, y),
         _diff(lambda t: so.SvLeverageExact.from_theta(t).score_first(nxt, y), theta, 1e-5)),
    )
    for name, got, want in cases:
        assert np.max(np.abs(got - want)) <= 1e-7 * max(1.0, np.max(np.abs(want))), (name, got - want)
    # the first pair's mu component is the total derivative, not score_main's partial at curr = mu
    assert not np.allclose(m.score_first(nxt, y)[0], m.score_main(np.full_like(nxt, m.mu), nxt, y)[0])


@pytest.mark.parametrize("lag", [3, 10, 25])
@pytest.mark.parametrize("pset", [0, 2])
def test_quadrature_reproduces_kalman(pset, lag):
    p = gi.LG_PARAM_SETS[pset]
    obs = gi.lg_obs(25, p, seed=11 + pset)
    q = sq.quadrature_targets(gp.LinearGaussian(p), p[1], obs, lag, -10.0, 10.0, m=1001, pair_y=1)
    k = km.fixed_lag_targets(obs, *p[:3], lag)
    ll = gp.kalman_loglike(obs, *p[:3])
    assert abs(q["log_like"] - ll) <= 1e-11 * abs(ll)
    assert np.max(np.abs(q["filt"] - km.filtered_means(obs, *p[:3]))) <= 1e-11 * np.max(np.abs(q["filt"]))
    assert np.max(np.abs(q["smo"] - k["smo"])) <= 1e-11 * np.max(np.abs(k["smo"]))
    # kalman.py's slot t + 1 = the pair (x_t, x_t+1)
    assert np.max(np.abs(q["score"][:3, :-1] - k["grad"][:, 1:])) <= 1e-11 * np.max(np.abs(k["grad"]))


@pytest.mark.parametrize("pset", [0, 1, 2])
def test_quadrature_fisher_identity_for_sv(pset):
    """lag = n_obs: every pair is conditioned on the whole series, so the score slots sum to d log_like / d theta; the
    first pair's total derivative is part of it"""
    params, theta = gi.SV_PARAM_SETS[pset], THETA[pset]
    obs = gi.sv_obs(20, params, seed=5 + pset)
    m, sd = _make(theta)
    lo, hi = params[0] - 8.0, params[0] + 8.0
    q = sq.quadrature_targets(m, sd, obs, 20, lo, hi, m=801, pair_y=0)
    fd = sq.fd_gradient(_make, theta, obs, lo, hi, m=801)
    assert np.max(np.abs(q["score"].sum(axis=1) - fd)) <= 1e-6 * np.max(np.abs(fd)), (q["score"].sum(axis=1), fd)
    # score_main in place of score_first for the pair (x_0, x_1) breaks it
    m2 = so.SvLeverageExact.from_theta(theta)
    m2.score_first = lambda x1, y0: m2.score_main(np.full_like(x1, m2.mu), x1, y0)
    q2 = sq.quadrature_targets(m2, sd, obs, 20, lo, hi, m=801, pair_y=0)
    assert abs(q2["score"].sum(axis=1)[0] - fd[0]) > 1e-3 * abs(fd[0]) + 1e-6


@pytest.mark.parametrize("pset", [0, 1])
def test_quadrature_louis_identity_for_sv(pset):
    """lag = n_obs: the summed hess1 and hess2 targets minus g g' equal the finite-difference Hessian of log_like, which
    checks the hess2 targets (the alpha recursion over the backward kernels)"""
    params, theta = gi.SV_PARAM_SETS[pset], THETA[pset]
    obs = gi.sv_obs(15, params, seed=9)
    m, sd = _make(theta)
    lo, hi = params[0] - 8.0, params[0] + 8.0
    q = sq.quadrature_targets(m, sd, obs, 15, lo, hi, m=401, pair_y=0, hessian=True)
    g = q["score"].sum(axis=1)
    h = q["hess1"].sum(axis=0) + q["hess2"].sum(axis=0) - np.outer(g, g)
    fd = sq.fd_hessian(_make, theta, obs, lo, hi, m=401)
    assert np.max(np.abs(h - fd)) <= 1e-5 * np.max(np.abs(fd)), (h, fd)


@pytest.mark.parametrize("lag", [2, 10])
def test_replay_reproduces_the_models_4_and_6_restatements(lag):
    p = gi.LG_PARAM_SETS[1]
    n, nobs = 300, 30
    obs = gi.lg_obs(nobs + 1, p, seed=77)[1:]
    rvr, rvp = gi.split_particle(gi.sv_rvs(n, nobs, 3), nobs)
    out = gp.flps_generic(gp.LinearGaussianFullyAdapted(p), obs, rvr, rvp, n, lag, dumps=True)
    model = fh.LinearGaussianFullyAdaptedHess(p)
    g, h1, h2 = so.predictive_replay(model, obs, out["X"], out["A"], out["W"], lag, hessian=True)
    assert np.array_equal(g, fo.predictive_gradient(model, obs, out["X"], out["A"], out["W"], lag))
    w1, w2 = fh.predictive_hessian(model, obs, out["X"], out["A"], out["W"], lag)
    assert np.max(np.abs(h1 - w1)) <= 1e-13 * np.max(np.abs(w1))
    assert np.max(np.abs(h2 - w2)) <= 1e-13 * np.max(np.abs(w2))


def test_restatement_gradient_against_quadrature_and_the_reference_pairings_bias():
    """n_obs = 30, lag 10, N = 1000, 60 replicates at the data-generating values (rho = -0.5): model 8's per-slot
    gradient has |z| <= 5 against the exact targets; model 0's (Q5 / Q6) summed gradient misses them by far more"""
    params, theta = gi.SV_PARAM_SETS[0], THETA[0]
    nobs, lag, n, reps = 30, 10, 1000, 60
    obs = gi.sv_obs(nobs, params, seed=321)
    m, sd = _make(theta)
    q = sq.quadrature_targets(m, sd, obs, lag, params[0] - 7.0, params[0] + 7.0, m=601, pair_y=0)
    g8, g0 = [], []
    for r in range(reps):
        rvr, rvp = gi.split_particle(gi.sv_rvs(n, nobs, 1000 + r), nobs)
        g8.append(so.flps_sv_exact(params, obs, rvr, rvp, n, lag)["gradient"])
        g0.append(gp.flps_generic(gp.SvLeverage(params), obs, rvr, rvp, n, lag)["gradient"])
    g8, g0 = np.array(g8), np.array(g0)
    s = g8.std(axis=0, ddof=1)
    live = s > 0.0
    z8 = (g8.mean(axis=0) - q["score"])[live] / (s[live] / np.sqrt(reps))
    assert np.all(q["score"][~live] == 0.0)      # slot n_obs - 1 and the atanh phi row of slot 0
    sums = {}
    for name, g in (("model 8", g8), ("model 0", g0)):
        gs = g.sum(axis=2)
        sums[name] = (gs.mean(axis=0) - q["score"].sum(axis=1)) / (gs.std(axis=0, ddof=1) / np.sqrt(reps))
        print(name, "summed gradient", np.round(gs.mean(axis=0), 3).tolist(), "exact",
              np.round(q["score"].sum(axis=1), 3).tolist(), "z", np.round(sums[name], 1).tolist())
    print("model 8 per-slot max |z|", np.max(np.abs(z8)))
    assert np.max(np.abs(z8)) <= 5.0
    assert np.all(np.abs(sums["model 8"]) <= 5.0)
    assert np.max(np.abs(sums["model 0"])) >= 20.0
