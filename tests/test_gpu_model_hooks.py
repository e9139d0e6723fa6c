"""Model-generic device hooks (csrc/pf_model.cuh, pmmh_flps_model_corr): the chain kernel instantiated
for (0) the reference's SV model -- bit-identical to pmmh_flps_sv_corr -- and (1) a linear Gaussian state
space model, checked against the NumPy restatement of the same algorithm with that model's callbacks
(oracle/generic_pf.py: ancestors exact, log-likelihood 1e-10, gradient 1e-9, the SV tolerances) and
against the exact Kalman likelihood."""
import numpy as np
import pytest

import golden_inputs as gi
from helpers import first_mismatch_step, relerr, to_time_major

pytestmark = pytest.mark.gpu


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def test_sv_through_the_generic_entry_is_bit_identical(cuda_dev):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    n, nobs, lag, B = 4096, 160, 10, 5
    obs = gi.sv_obs(nobs)
    rs = np.random.RandomState(3)
    params = np.array(gi.SV_PARAM_SETS[0]) + 0.01 * rs.normal(size=(B, 4))
    u = rs.normal(size=(B, nobs, n))
    rvr = rs.uniform(size=(B, nobs))
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, params, rvr, u)
    a = K.flps_model_corr(_lib.MODEL_SV_LEVERAGE, obs_d, par_d, rvr_d, u_d, lag=lag)
    K.set_sv_algorithm(3)          # the chain kernel behind pmmh_flps_sv_corr, no fallback pass
    try:
        b = K.flps_sv_corr(obs_d, par_d, rvr_d, u_d, lag=lag, compute_hessian=False)
        torch.cuda.synchronize()
    finally:
        K.set_sv_algorithm(0)
    assert int(b["diag"][0, 6]) == 3 and int(a["diag"][:, 2].max()) == 0
    for k in ("log_like", "filt", "smo", "gradient", "traj"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("n,nobs,lag,seed", [(500, 150, 10, 0), (4096, 200, 10, 1), (1000, 100, 4, 2), (75, 361, 10, 0),
                                             (333, 90, 2, 1), (1000, 100, 4, 3), (64, 60, 10, 3)])
def test_linear_gaussian_vs_generic_oracle(cuda_dev, n, nobs, lag, seed):
    import torch
    import generic_pf as gp
    from pmmh_qn_b200 import _lib, kernels as K
    obs, params, rvr, rvp = gi.lg_inputs(n, nobs, seed)
    ref = gp.flps_generic(gp.LinearGaussian(params), obs, rvr, rvp, n, lag, dumps=True)
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, params, rvr[:nobs], to_time_major(rvp, n, nobs))
    out = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr_d, u_d, lag=lag, store_history=True)
    torch.cuda.synchronize()
    assert int(out["diag"][0, 2]) == 0
    A = out["A"][0].cpu().numpy()
    step = first_mismatch_step(A[1:], ref["A"][1:])
    assert step is None, "ancestors differ first at time %d (near ties %d)" % (step + 1, int(out["diag"][0, 0]))
    assert relerr(out["X"][0].cpu().numpy(), ref["X"]) <= 1e-12
    ll = float(out["log_like"][0])
    assert abs(ll - ref["log_like"]) <= 1e-10 * abs(ref["log_like"])
    assert relerr(out["filt"][0].cpu().numpy(), ref["filt"]) <= 1e-10
    assert relerr(out["smo"][0].cpu().numpy(), ref["smo"]) <= 1e-10
    g = out["gradient"][0].cpu().numpy()
    assert np.max(np.abs(g - ref["gradient"])) <= 1e-9 * np.max(np.abs(ref["gradient"]))
    assert np.all(g[3] == 0.0)


def test_linear_gaussian_likelihood_against_the_kalman_filter(cuda_dev):
    """The particle estimate of the log-likelihood is consistent with the exact value (N = 4096, T = 200,
    16 independent u; the estimator of the LOG-likelihood is biased by about -var/2): every estimate within
    2.5, the mean within 4 standard errors + 0.25."""
    import generic_pf as gp
    from pmmh_qn_b200 import _lib, kernels as K
    n, nobs, B = 4096, 201, 16
    params = np.array(gi.LG_PARAM_SETS[0])
    obs = gi.lg_obs(nobs, params)
    exact = gp.kalman_loglike(obs, *params[:3])
    rs = np.random.RandomState(12)
    u = rs.normal(size=(B, nobs, n))
    rvr = rs.uniform(size=(B, nobs))
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, np.tile(params, (B, 1)), rvr, u)
    out = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr_d, u_d, lag=10)
    ll = out["log_like"].cpu().numpy()
    assert np.all(np.abs(ll - exact) < 2.5), (ll, exact)
    assert abs(ll.mean() - exact) < 4.0 * ll.std(ddof=1) / np.sqrt(B) + 0.25, (ll.mean(), exact, ll.std())


def test_fully_adapted_filter_against_the_kalman_filter(cuda_dev):
    """PMMH_MODEL_LINEAR_GAUSSIAN_FA: optimal proposal + predictive weights through the same kernel (shifted
    observations).  log p(y_1) + its estimate of log p(y_2..y_T | y_1) is consistent with the exact value and
    much less variable than the bootstrap filter's estimate on the same data and u."""
    import generic_pf as gp
    from pmmh_qn_b200 import _lib, kernels as K
    n, nobs, B = 4096, 201, 16
    params = np.array(gi.LG_PARAM_SETS[0])
    phi, sv, se = params[:3]
    obs = gi.lg_obs(nobs, params)
    exact = gp.kalman_loglike(obs, phi, sv, se)
    ll_y1 = gp.log_p_y1(obs, sv, se)
    rs = np.random.RandomState(12)
    u = rs.normal(size=(B, nobs, n))
    rvr = rs.uniform(size=(B, nobs))
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, np.tile(params, (B, 1)), rvr, u)
    boot = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr_d, u_d, lag=10)["log_like"].cpu().numpy()
    shifted = np.ascontiguousarray(obs[1:])                                    # obs'[t] = obs[t + 1]
    obs_s, rvr_s, u_s = _dev(cuda_dev, shifted, rvr[:, :nobs - 1], u[:, :nobs - 1])
    out = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA, obs_s, par_d, rvr_s, u_s, lag=10)
    assert int(out["diag"][:, 2].max()) == 0
    fa = out["log_like"].cpu().numpy() + ll_y1
    assert np.all(np.abs(fa - exact) < 0.5), (fa, exact)
    assert abs(fa.mean() - exact) < 4.0 * fa.std(ddof=1) / np.sqrt(B) + 0.05, (fa.mean(), exact, fa.std())
    assert fa.std(ddof=1) < 0.5 * boot.std(ddof=1), (fa.std(ddof=1), boot.std(ddof=1))
    assert np.all(out["gradient"].cpu().numpy() == 0.0)


def test_generic_entry_rejects_bad_arguments(cuda_dev):
    from pmmh_qn_b200 import _lib, kernels as K
    obs, params, rvr, rvp = gi.lg_inputs(100, 40, 0)
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, params, rvr[:40], to_time_major(rvp, 100, 40))
    with pytest.raises(_lib.PmmhError):
        K.flps_model_corr(7, obs_d, par_d, rvr_d, u_d, lag=10)
    with pytest.raises(_lib.PmmhError):
        K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr_d, u_d, lag=11)
