"""The sort-edge inputs of tests/sort_edge_inputs.py are what they claim, by construction and through the oracles
(C oracle for SV, oracle/generic_pf.py for the linear Gaussian models, tests/fa_gradient_oracle.py for model 4),
which run on every pattern at small N and give finite outputs."""
import numpy as np
import pytest

import golden_inputs as gi
import sort_edge_inputs as se

N, NOBS, LAG = 600, 24, 10
SV = (0.2, 0.9, 0.4, -0.5)


def _oracle(params, u, rvp, seed, hessian=0):
    import oracle
    rvr = gi.split_particle(gi.sv_rvs(u.shape[1], u.shape[0], seed), u.shape[0])[0]
    return oracle.flps_sv_corr(gi.sv_obs(u.shape[0]), np.array(params), rvr, rvp, u.shape[1], LAG, hessian,
                               dumps=True)


def test_layouts_agree():
    u, rvp = se.build("plain", 7, 5, 0)
    for t in range(5):
        for j in range(7):
            assert rvp[t + j * 5] == u[t, j]


@pytest.mark.parametrize("m", [2, 16])
def test_sibling_ties(m):
    u, rvp = se.build("sibling_ties", N, NOBS, 1, m=m)
    for t in range(1, NOBS):
        if t >= 2 and t % 2 == 0:
            assert np.all(u[t] == np.repeat(u[t, ::m], m)[:N]), t
        else:
            assert np.unique(u[t]).size == N, t
    ref = _oracle(SV, u, rvp, 1, hessian=1)
    X, A = ref["X"], ref["A"]
    ties = 0
    for t in range(1, NOBS):
        eq = np.nonzero(np.diff(X[t]) == 0.0)[0]
        if t % 2 == 1:
            assert eq.size == 0, t
        # every tie is between children of one parent
        assert np.all(A[t][eq] == A[t][eq + 1]), t
        ties += eq.size
    assert ties > 0
    for k in ("log_like", "filt", "smo", "gradient", "hess1", "hess2"):
        assert np.all(np.isfinite(ref[k])), k


@pytest.mark.parametrize("g", [2, 3, 300])
def test_tie_group(g):
    u, rvp = se.build("tie_group", N, NOBS, 2, g=g)
    assert np.sum(u[1] == se.GROUP_U) == g
    rest = u[1][u[1] != se.GROUP_U]
    assert np.all(np.abs(rest) < se.TRUNC)
    ref = _oracle(SV, u, rvp, 2)
    x1 = ref["X"][1]
    top = x1[-g:]
    assert np.all(top == top[0]) and x1[-g - 1] < top[0]
    assert np.unique(x1[:-g]).size == N - g
    for k in ("log_like", "filt", "smo", "gradient"):
        assert np.all(np.isfinite(ref[k])), k


def test_tie_group_is_the_only_content_of_its_bin():
    """1 sd of the propagation clear of everything else of its row: alone in any bin of width <= 1 sd"""
    u, rvp = se.build("tie_group", N, NOBS, 3, g=5)
    ref = _oracle(SV, u, rvp, 3)
    sd = se.sv_child_sd(SV)
    x1 = ref["X"][1]
    assert x1[-5] - x1[-6] > (se.GROUP_U - se.TRUNC) * sd * (1.0 - 1e-12)


def test_outliers():
    u, rvp = se.build("outliers", N, NOBS, 4)
    for t in range(1, NOBS):
        assert u[t, 0] == -40.0 and u[t, N - 1] == 40.0
        assert sorted(u[t][np.abs(u[t]) >= 7.0]) == sorted(se.OUTLIER_U)
    ref = _oracle(SV, u, rvp, 4, hessian=1)
    sd = se.sv_child_sd(SV)
    X = ref["X"]
    for t in range(1, NOBS):
        # the extreme children sit at sorted positions 0 and N - 1, far outside the rest of the cloud
        assert X[t][1] - X[t][0] > 20.0 * sd and X[t][-1] - X[t][-2] > 20.0 * sd, t
        assert np.unique(X[t]).size == N
    for k in ("log_like", "filt", "smo", "gradient", "hess1", "hess2"):
        assert np.all(np.isfinite(ref[k])), k


@pytest.mark.parametrize("m", [2, 4])
def test_near_ties(m):
    sd, xs = se.sv_child_sd(SV), se.sv_xscale(SV)
    u, rvp = se.build("near_ties", N, NOBS, 5, m=m, sd=sd, xscale=xs)
    ref = _oracle(SV, u, rvp, 5, hessian=1)
    X, A = ref["X"], ref["A"]
    near = 0
    for t in range(1, NOBS):
        d = np.diff(X[t])
        assert np.all(d > 0.0), t          # no exact tie anywhere
        sib = A[t][1:] == A[t][:-1]
        near += int(np.sum(sib & (d <= 4 * np.spacing(xs))))
        assert np.max(np.abs(X[t])) < xs
    assert near > NOBS     # near-tied siblings at most steps
    for k in ("log_like", "filt", "smo", "gradient", "hess1", "hess2"):
        assert np.all(np.isfinite(ref[k])), k


@pytest.mark.parametrize("sigma_v", [1e-4, 1e-8])
def test_narrow_cloud_oracles(sigma_v):
    import generic_pf as gp
    import fa_gradient_oracle as fo
    u, rvp = se.build("plain", N, NOBS, 6)
    ref = _oracle((0.2, 0.9, sigma_v, -0.5), u, rvp, 6, hessian=1)
    assert np.all(np.diff(ref["X"][1:], axis=1) > 0.0)
    for k in ("log_like", "filt", "smo", "gradient", "hess1", "hess2"):
        assert np.all(np.isfinite(ref[k])), k
    rvr = gi.split_particle(gi.sv_rvs(N, NOBS, 6), NOBS)[0]
    lg = (0.8, sigma_v, 0.3, 0.0)
    obs = gi.lg_obs(NOBS, gi.LG_PARAM_SETS[0])
    for model, ob in ((gp.LinearGaussian(lg), obs), (gp.LinearGaussianFullyAdapted(lg), obs[1:])):
        r = gp.flps_generic(model, ob, rvr, se.build("plain", N, ob.shape[0], 6)[1], N, LAG)
        assert np.isfinite(r["log_like"]) and np.all(np.isfinite(r["gradient"]))
    r = fo.flps_fa_grad(np.array(lg), obs[1:], rvr, se.build("plain", N, NOBS - 1, 6)[1], N, LAG)
    assert np.isfinite(r["log_like"]) and np.all(np.isfinite(r["gradient"]))


@pytest.mark.parametrize("pattern", ["sibling_ties", "tie_group", "outliers", "near_ties"])
def test_model_oracles_finite(pattern):
    import generic_pf as gp
    import fa_gradient_oracle as fo
    params = np.array(gi.LG_PARAM_SETS[0])
    obs = gi.lg_obs(NOBS + 1, gi.LG_PARAM_SETS[0])
    rvr = gi.split_particle(gi.sv_rvs(N, NOBS, 7), NOBS)[0]
    kw = dict(m=4, g=7, sd=params[1], xscale=8.0)
    _, rvp = se.build(pattern, N, NOBS, 7, **kw)
    for model, ob in ((gp.LinearGaussian(params), obs[:NOBS]), (gp.LinearGaussianFullyAdapted(params), obs[1:])):
        r = gp.flps_generic(model, ob, rvr, rvp, N, LAG)
        assert np.isfinite(r["log_like"]) and np.all(np.isfinite(r["gradient"])) and np.all(np.isfinite(r["smo"]))
    r = fo.flps_fa_grad(params, obs[1:], rvr, rvp, N, LAG)
    assert np.isfinite(r["log_like"]) and np.all(np.isfinite(r["gradient"]))


def test_rounding_ties_differ_from_the_reference_only_in_order():
    """At sigma_v = 1e-8, N = 2^14 children meet exact ties by rounding, between children of different parents of
    different values.  glibc's merge sort (the C oracle's qsort) puts them in descending birth order, the stable sort of
    oracle/generic_pf.py in ascending birth order, as the kernels do: the generations are the same values, the
    ancestors differ only inside runs of equal children, and the estimates agree to 1e-12."""
    import generic_pf as gp
    import oracle
    n, nobs = 1 << 14, 40
    params = np.array((SV[0], SV[1], 1e-8, SV[3]))
    u, rvp = se.build("plain", n, nobs, 11)
    obs, rvr = gi.sv_obs(nobs), gi.split_particle(gi.sv_rvs(n, nobs, 11), nobs)[0]
    ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, LAG, 0, dumps=True)
    res = gp.flps_generic(gp.SvLeverage(params), obs, rvr, rvp, n, LAG, dumps=True)
    assert np.array_equal(ref["X"], res["X"])
    rows = np.nonzero(np.any(ref["A"] != res["A"], axis=1))[0]
    assert rows.size > 0
    for t in rows:
        x = ref["X"][t]
        runs = np.split(np.arange(n), np.nonzero(np.diff(x))[0] + 1)
        for r in runs:
            if not np.array_equal(ref["A"][t][r], res["A"][t][r]):
                assert r.size > 1 and np.all(x[r] == x[r[0]]), t
                assert np.array_equal(np.sort(ref["A"][t][r]), np.sort(res["A"][t][r])), t
                assert np.all(np.diff(res["A"][t][r]) >= 0) and np.all(np.diff(ref["A"][t][r]) <= 0), t
    assert abs(res["log_like"] - ref["log_like"]) <= 1e-12 * abs(ref["log_like"])
    for k in ("filt", "smo", "traj", "gradient"):
        assert np.max(np.abs(res[k] - ref[k])) <= 1e-12 * np.max(np.abs(ref[k])), k
