"""Data and parameter edges of the kernels that shift the log-weights by a bound instead of their maximum.

The reference shifts by one of the log-weights (Q4); the chain, exchange, streaming and grid kernels shift by the
largest log-weight over a PREDICTED child range (chain and streaming: the extreme propagation means widened by
6.5 sd; exchange: the weighted moments of the propagation means; grid: the occupied histogram bins).  Any shift
cancels, as long as it does not drift so far above the true maximum (about 700 log units) that the weights become
subnormal or 0.  The gap grows with an observation far out in the tail and with parameters far from the data (a
NumPy simulation of the chain kernel's rule, SV, mu = -6, a 12 sd outlier: about 170), and the SV log-weight has
its own branch for y = 0 (log y^2 = -inf).  Every case is compared with the C oracle (SV) or oracle/generic_pf.py (linear Gaussian,
bootstrap and fully adapted), at the suite's SV tolerances:

- the SV entry pmmh_flps_sv_corr under algorithms 1, 2, 3, 5 and 6 (N = 5000; N = 1000 on the chain kernel);
- the model entry pmmh_flps_model_corr for models 0, 1 and 2 on the chain kernel (N = 1000) and the grid kernel
  (N = 5000);

on series with exact zeros (t = 1, the middle, inside the last lag steps), a 12 sd outlier (the middle, the last
lag steps), and SV parameters far from the data (mu = -4, -6), without leverage (rho = 0), with rho = +-0.95 and
phi = 0.  The grid and exchange kernels may abandon an evaluation (diag[PMMH_DIAG_STATUS] == 1); on the SV entry
algorithm 0 then reruns it on the general kernel, whose outputs must match the oracle.
"""
import numpy as np
import pytest

import golden_inputs as gi
from helpers import first_mismatch_step, relerr, to_time_major

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_SOFT_TIES, DIAG_KERNEL = 2, 4, 6
CHAIN, GRID = 3, 5
NOBS, LAG = 80, 10
SERIES = ["plain", "zero_first", "zero_mid", "zero_tail", "outlier_mid", "outlier_tail"]
SV_EDGE_PARAMS = {
    "base": (0.2, 0.9, 0.4, -0.5),
    "mu-4": (-4.0, 0.9, 0.4, -0.5),
    "mu-6": (-6.0, 0.9, 0.4, -0.5),
    "rho0": (0.2, 0.9, 0.4, 0.0),
    "rho+0.95": (0.2, 0.9, 0.4, 0.95),
    "rho-0.95": (0.2, 0.9, 0.4, -0.95),
    "phi0": (0.2, 0.0, 0.4, -0.5),
}
LG_EDGE_PARAMS = {"lg%d" % i: p for i, p in enumerate(gi.LG_PARAM_SETS)}
FA_EDGE_PARAMS = dict(LG_EDGE_PARAMS, unit_root=(0.999, 0.05, 1.0, 0.0))
# the kernel each algorithm of pmmh_sv_set_algorithm runs at these sizes (streaming kernels report 4)
SV_KERNEL_OF = {1: 1, 2: 2, 3: CHAIN, 5: 4, 6: GRID}


def _edge(y, kind):
    """y with one edge: an exact zero or a 12 sd outlier at t = 1, in the middle, or inside the last LAG steps"""
    y = np.array(y, dtype=np.float64)
    at = {"first": 1, "mid": len(y) // 2, "tail": len(y) - LAG // 2}
    if kind.startswith("zero_"):
        y[at[kind[5:]]] = 0.0
    elif kind.startswith("outlier_"):
        y[at[kind[8:]]] = 12.0 * np.std(y)
    return y


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def _check(res, ref, exact_zero_gradient=False, grid=False):
    """one problem's device outputs (NumPy) against the reference at the SV tolerances; with the history, ancestors
    exact, except that on the grid kernel a first differing generation may come with a counted soft tie, and the
    outputs then agree up to it"""
    if "A" in res:
        step = first_mismatch_step(res["A"][1:], ref["A"][1:])
        if step is not None:
            assert grid, "ancestors differ first at time %d" % (step + 1)
            assert int(res["diag"][DIAG_SOFT_TIES]) > 0, "ancestors differ first at time %d" % (step + 1)
            assert relerr(res["X"][:step + 1], ref["X"][:step + 1]) <= 1e-12
            assert relerr(res["filt"][:step + 1], ref["filt"][:step + 1]) <= 1e-10
            return
        assert relerr(res["X"], ref["X"]) <= 1e-12
    assert np.isfinite(ref["log_like"])
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"]), (res["log_like"], ref["log_like"])
    assert relerr(res["filt"], ref["filt"]) <= 1e-10
    assert relerr(res["smo"], ref["smo"]) <= 1e-10
    assert relerr(res["traj"], ref["traj"]) <= 1e-12
    g = res["gradient"]
    if exact_zero_gradient:
        assert np.all(g == 0.0)
    else:
        assert np.max(np.abs(g - ref["gradient"])) <= 1e-9 * np.max(np.abs(ref["gradient"]))


@pytest.mark.parametrize("pname", list(SV_EDGE_PARAMS))
@pytest.mark.parametrize("series", SERIES)
@pytest.mark.parametrize("alg", sorted(SV_KERNEL_OF))
def test_sv_entry_edges_vs_oracle(cuda_dev, alg, series, pname):
    import oracle
    import torch
    from pmmh_qn_b200 import kernels as K
    n = 1000 if alg == 3 else 5000
    obs = _edge(gi.sv_obs(NOBS), series)
    params = np.array(SV_EDGE_PARAMS[pname])
    rvr, rvp = gi.split_particle(gi.sv_rvs(n, NOBS, 9), NOBS)
    ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, LAG, 0)
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, params, rvr, to_time_major(rvp, n, NOBS))

    def run(a):
        K.set_sv_algorithm(a)
        try:
            out = K.flps_sv_corr(obs_d, par_d, rvr_d, u_d, lag=LAG, compute_hessian=False)
            torch.cuda.synchronize()
        finally:
            K.set_sv_algorithm(0)
        return {k: v[0].cpu().numpy() for k, v in out.items() if not k.startswith("_")}

    res = run(alg)
    d = res["diag"]
    assert int(d[DIAG_KERNEL]) == SV_KERNEL_OF[alg], d
    if int(d[DIAG_STATUS]) == 1 and alg in (2, 6):
        # the grid and exchange kernels may give up on a cloud their fixed-capacity layout does not hold; the
        # automatic selection then reruns the evaluation on the general kernel
        res = run(0)
        assert int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
    else:
        assert int(d[DIAG_STATUS]) == 0, d
    _check(res, ref)


MODEL_CASES = ([(0, k) for k in SV_EDGE_PARAMS] + [(1, k) for k in LG_EDGE_PARAMS] +
               [(2, k) for k in FA_EDGE_PARAMS])


@pytest.mark.parametrize("model_id,pname", MODEL_CASES, ids=["m%d-%s" % c for c in MODEL_CASES])
@pytest.mark.parametrize("series", SERIES)
@pytest.mark.parametrize("kernel", [CHAIN, GRID])
def test_model_entry_edges_vs_reference(cuda_dev, kernel, series, model_id, pname):
    import generic_pf as gp
    import oracle
    from pmmh_qn_b200 import kernels as K
    n = 1000 if kernel == CHAIN else 5000
    rvr, rvp = gi.split_particle(gi.sv_rvs(n, NOBS, 10 + model_id), NOBS)
    if model_id == 0:
        params = np.array(SV_EDGE_PARAMS[pname])
        obs = _edge(gi.sv_obs(NOBS), series)
        ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, LAG, 0, dumps=True)
    else:
        params = np.array((LG_EDGE_PARAMS if model_id == 1 else FA_EDGE_PARAMS)[pname])
        if model_id == 1:
            obs = _edge(gi.lg_obs(NOBS, gi.LG_PARAM_SETS[0]), series)
            model = gp.LinearGaussian(params)
        else:   # the fully adapted filter takes the shifted series obs'[t] = obs[t + 1]
            obs = _edge(gi.lg_obs(NOBS + 1, gi.LG_PARAM_SETS[0])[1:], series)
            model = gp.LinearGaussianFullyAdapted(params)
        ref = gp.flps_generic(model, obs, rvr, rvp, n, LAG, dumps=True)
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, params, rvr, to_time_major(rvp, n, NOBS))
    out = K.flps_model_corr(model_id, obs_d, par_d, rvr_d, u_d, lag=LAG, store_history=True)
    res = {k: v[0].cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    d = res["diag"]
    assert int(d[DIAG_KERNEL]) == kernel, d
    if kernel == GRID and int(d[DIAG_STATUS]) == 1:
        # the model entry has no fallback pass: an evaluation the grid kernel gives up on is reported through
        # diag[PMMH_DIAG_STATUS] and its outputs are not defined
        return
    assert int(d[DIAG_STATUS]) == 0, d
    _check(res, ref, exact_zero_gradient=model_id == 2, grid=kernel == GRID)
