"""CPU: pin the oracle (oracle/pmmh_oracle.c) bit-for-bit against the golden vectors that were
produced by the reference's own compiled Cython kernels (tests/golden/make_golden.py), and --
when oracle/_ref is present -- against the compiled reference directly on fresh inputs."""
import os
import sys

import numpy as np
import pytest

import golden_inputs as gi
import oracle


def _same(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64).reshape(a.shape)
    return np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("case", gi.SV_KERNEL_CASES, ids=lambda c: "n%d_t%d_l%d" % c[:3])
def test_flps_and_bpf_bit_exact_vs_golden(golden, case):
    n, nobs, lag, seeds = case
    g = golden["sv_kernels"]
    for seed in seeds:
        obs, params, rvr, rvp = gi.sv_inputs(n, nobs, seed)
        tag = "n%d_t%d_l%d_s%d" % (n, nobs, lag, seed)
        for hess in (0, 1):
            o = oracle.flps_sv_corr(obs, params, rvr, rvp, n, lag, hess)
            pre = "flps_%s_h%d_" % (tag, hess)
            assert o["log_like"] == float(g[pre + "log_like"]) or (
                np.isnan(o["log_like"]) and np.isnan(g[pre + "log_like"]))
            for k in ("filt", "smo", "gradient", "traj", "hess1", "hess2"):
                assert _same(o[k], g[pre + k]), (tag, hess, k)
        if n <= 1024:
            o = oracle.bpf_sv_corr(obs, params, rvr, rvp, n)
            pre = "bpf_%s_" % tag
            assert _same(o["log_like"], g[pre + "log_like"])
            assert _same(o["filt"], g[pre + "filt"])
            assert _same(o["traj"], g[pre + "traj"])


def test_importance_discrete_bit_exact_vs_golden(golden):
    g = golden["re_kernels"]
    for (n, nobs, seeds) in gi.RE_KERNEL_CASES:
        for seed in seeds:
            obs, params, rvr, rvp = gi.re_inputs(n, nobs, seed)
            o = oracle.importance_discrete(obs, params, rvr, rvp, n)
            pre = "is_n%d_t%d_s%d_" % (n, nobs, seed)
            assert o["log_like"] == float(g[pre + "log_like"])
            for k in ("filt", "traj", "gradient"):
                assert _same(o[k], g[pre + k]), (pre, k)


def test_stratified_exact_vs_golden(golden):
    g = golden["ss_kernels"]
    for (m, n, seeds) in gi.SS_KERNEL_CASES:
        for seed in seeds:
            r = gi.ss_inputs(m, seed)
            assert np.array_equal(oracle.stratified(r, n), g["strat_m%d_n%d_s%d" % (m, n, seed)])


def test_estimator_level_postprocessing_vs_golden(golden):
    """smoother_post (cython.py:100-126 incl. the Q9 scalar np.inner) reproduces the reference
    estimator's log_joint_gradient_estimate / hessian before priors are added."""
    g = golden["estimators"]
    n, nobs, lag = 75, 361, 10
    for ci, params in enumerate(gi.SV_ESTIMATOR_PARAMS):
        rvs = gi.sv_rvs(n, nobs, seed=1000 + ci)
        rvr, rvp = oracle.split_rvs_particle(rvs, nobs)
        obs = gi.sv_obs(nobs)
        for hess in (0, 1):
            o = oracle.flps_sv_corr(obs, np.array(params), rvr, rvp, n, lag, hess)
            grad_est, hess_est = oracle.smoother_post(o["gradient"], o["hess1"], o["hess2"], hess)
            pre = "sv_smoother_c%d_h%d_" % (ci, hess)
            assert o["log_like"] == float(g[pre + "log_like"])
            # the golden gradient estimate already has the prior gradient added in place
            # (base_state_inference.py:71); remove it again
            assert np.allclose(grad_est + g[pre + "prior_grad"], g[pre + "log_joint_gradient_estimate"],
                               rtol=0, atol=1e-12 * np.max(np.abs(grad_est)))
            if hess:
                want = g[pre + "log_joint_hessian_estimate"] + np.diag(g[pre + "prior_hess"])
                assert np.allclose(hess_est, want, rtol=1e-12, atol=1e-9)


def test_logistic_oracle_vs_golden(golden):
    g = golden["estimators"]
    n_data, d, m = 110000, gi.LOGIT_D, 5500
    x, y, beta = gi.logit_data(n_data, d)
    for ci in range(2):
        u = gi.logit_u(m, seed=3000 + ci)
        idx = oracle.subsample_indices(u, n_data)
        for hess in (0, 1):
            o = oracle.logistic_loglike_gradient(beta, x, y, idx, True, bool(hess))
            pre = "logit_smoother_c%d_h%d_" % (ci, hess)
            assert abs(o["log_like"] - float(g[pre + "log_like"])) <= 1e-12 * abs(o["log_like"])
            assert np.allclose(o["gradient"], g[pre + "gradient"], rtol=1e-11, atol=1e-11)
            if hess:
                assert np.allclose(o["hessian"], g[pre + "hessian"], rtol=1e-10, atol=1e-9)


@pytest.mark.skipif(not os.path.isdir(os.path.join(os.path.dirname(oracle.__file__), "_ref")),
                    reason="oracle/_ref not built")
def test_oracle_vs_compiled_reference_fresh_inputs():
    """Bit-exact against the compiled reference itself on inputs that are not in the goldens."""
    import build_ref
    for (n, nobs, lag) in [(75, 361, 10), (200, 120, 10), (64, 40, 4)]:
        ref = build_ref.load("sv", n, nobs, lag)
        if ref is None:
            pytest.skip("variant not built")
        rs = np.random.RandomState(777 + n)
        obs = gi.sv_obs(nobs, seed=42)
        params = np.array([0.1, 0.93, 0.3, -0.4]) + 0.01 * rs.normal(size=4)
        rvr, rvp = oracle.split_rvs_particle(rs.normal(size=(nobs, n + 1)), nobs)
        for hess in (0, 1):
            r = ref.flps_sv_corr(obs, params, rvr, np.ascontiguousarray(rvp), hess)
            o = oracle.flps_sv_corr(obs, params, rvr, rvp, n, lag, hess)
            for k, name in enumerate(("filt", "smo", "log_like", "gradient", "traj", "hess1", "hess2")):
                assert _same(o[name], r[k]), (n, hess, name)
        r = ref.bpf_sv_corr(obs, params, rvr, np.ascontiguousarray(rvp))
        o = oracle.bpf_sv_corr(obs, params, rvr, rvp, n)
        assert _same(o["filt"], r[0]) and _same(o["log_like"], r[1]) and _same(o["traj"], r[2])


def test_generic_numpy_restatement_reproduces_the_c_oracle():
    """oracle/generic_pf.py (the checker of the model-generic device entry point) with the SV callbacks
    = oracle_flps_sv_corr: ancestors and sorted generations exact, estimates to 1e-12."""
    import generic_pf as gp
    import oracle
    for (n, nobs, lag, seed) in [(75, 361, 10, 0), (200, 120, 10, 1), (64, 40, 4, 0), (37, 50, 10, 1)]:
        obs, params, rvr, rvp = gi.sv_inputs(n, nobs, seed)
        ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, lag, 0, dumps=True)
        got = gp.flps_generic(gp.SvLeverage(params), obs, rvr, rvp, n, lag, dumps=True)
        assert np.array_equal(got["A"][1:], ref["A"][1:])
        for k in ("X", "filt", "smo", "gradient"):
            assert np.max(np.abs(got[k] - ref[k])) <= 1e-12 * np.max(np.abs(ref[k])), k
        assert abs(got["log_like"] - ref["log_like"]) <= 1e-12 * abs(ref["log_like"])
        assert np.max(np.abs(got["traj"][1:] - ref["traj"][1:])) <= 1e-12 * np.max(np.abs(ref["traj"]))


@pytest.mark.parametrize("params", gi.LG_PARAM_SETS)
def test_fully_adapted_proposal_is_the_conditional_law(params):
    """generic_pf.LinearGaussianFullyAdapted (the checker of model id 2): propagate(xp, y, 0) and sdp^2 are the
    mean and variance of x_t given x_{t-1} = xp and y_t = y, written in precision-weighted form."""
    import generic_pf as gp
    phi, sv, se = params[:3]
    m = gp.LinearGaussianFullyAdapted(params)
    rs = np.random.RandomState(5)
    xp, y = 3.0 * rs.normal(size=1000), 3.0 * rs.normal(size=1000)
    prec = 1.0 / sv ** 2 + 1.0 / se ** 2
    mean = (phi * xp / sv ** 2 + y / se ** 2) / prec
    assert np.max(np.abs(m.propagate(xp, y, 0.0) - mean)) <= 1e-14 * np.max(np.abs(mean))
    assert abs(m.sdp ** 2 - 1.0 / prec) <= 1e-14 / prec


@pytest.mark.parametrize("params", gi.LG_PARAM_SETS)
def test_fully_adapted_restatement_against_the_kalman_filter(params):
    """log p(y_1) + flps_generic's estimate of log p(y_2 .. y_T | y_1) with the fully adapted callbacks on obs[1:] is
    the exact Kalman log-likelihood up to Monte Carlo error (N = 20000, T = 100: errors up to 0.06 were seen over
    3 seeds per set); its gradient rows are 0."""
    import generic_pf as gp
    phi, sv, se = params[:3]
    n, nobs = 20000, 101
    obs = gi.lg_obs(nobs, params)
    rvr, rvp = gi.split_particle(gi.sv_rvs(n, nobs - 1, 200), nobs - 1)
    r = gp.flps_generic(gp.LinearGaussianFullyAdapted(params), obs[1:], rvr, rvp, n, 10)
    exact = gp.kalman_loglike(obs, phi, sv, se)
    assert abs(r["log_like"] + gp.log_p_y1(obs, sv, se) - exact) < 0.25, (r["log_like"], exact)
    assert np.all(r["gradient"] == 0.0)
