"""Every SV smoother kernel against the C oracle at every lag (2 .. 63) and series length (down to n_obs = lag + 1) its
eligibility rule accepts, shapes from tests/sv_lag_edge_shapes.py.

Below n_obs = 2 lag - 1 the reference's tail indexes gradient slots < 0; the oracle and every kernel drop those terms
(DESIGN.md section 2), so besides the suite's bars -- ancestors exact, X and traj 1e-12, log-likelihood, filt and smo
1e-10, gradient 1e-9 |g|max, hess1 / hess2 1e-8 |H|max -- the exactly-zero gradient slots must be the oracle's.

Also: algorithm 0 at shapes the grid kernel refuses; the Philox, host-streamed and split-filter entries at lag 63; the
model entry on the chain kernel at lag + 1 <= n_obs < 2 lag (model 0 bit for bit with the SV entry, model 8 against its
restatement) and model 8's Hessian on the grid kernel at n_obs = 2 lag; and one step outside each kernel's rule, the
forced algorithm runs another kernel (which pins the rules of sv_lag_edge_shapes.py to the library's).
"""
import functools

import numpy as np
import pytest

import golden_inputs as gi
import sv_lag_edge_shapes as sh
from helpers import first_mismatch_step, relerr, to_time_major

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_KERNEL = 2, 6
GENERAL, EXCHANGE, CHAIN, STREAMING, GRID = 1, 2, 3, 4, 5
SV, SVX = 0, 8


@functools.lru_cache(maxsize=4)
def _host(n, nobs, lag):
    """(obs, params, rvr, rvp, u) of one shape; the parameter set cycles with the shape"""
    obs, params, rvr, rvp = gi.sv_inputs(n, nobs, 1000 + 7 * lag + nobs + n % 97)
    return obs, params, rvr, rvp, to_time_major(rvp, n, nobs)


@functools.lru_cache(maxsize=2)
def _oracle(n, nobs, lag, hess):
    import oracle
    obs, params, rvr, rvp, _ = _host(n, nobs, lag)
    return oracle.flps_sv_corr(obs, params, rvr, rvp, n, lag, hess, dumps=True)


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def _np(out, b=0):
    return {k: v[b].cpu().numpy() for k, v in out.items() if not k.startswith("_")}


def _run(cuda_dev, alg, n, nobs, lag, hess=0, hist=True, ctas=0):
    import torch
    from pmmh_qn_b200 import kernels as K
    obs, params, rvr, _, u = _host(n, nobs, lag)
    d = _dev(cuda_dev, obs, params, rvr, u)
    K.set_sv_algorithm(alg)
    try:
        out = K.flps_sv_corr(*d, lag=lag, compute_hessian=hess, store_history=hist, ctas_per_problem=ctas)
        torch.cuda.synchronize()
    finally:
        K.set_sv_algorithm(0)
    return _np(out)


def _check(res, ref, kernel, hessian=False):
    """kernel: the diag's kernel id, None where the entry reports none (the split filter)"""
    if kernel is not None:
        assert int(res["diag"][DIAG_KERNEL]) == kernel, res["diag"]
    assert int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
    if "A" in res:
        step = first_mismatch_step(res["A"][1:].astype(np.int64), ref["A"][1:].astype(np.int64))
        assert step is None, "ancestors differ first at time %d" % (step + 1)
        assert relerr(res["X"], ref["X"]) <= 1e-12
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"]), (res["log_like"],
                                                                                            ref["log_like"])
    assert relerr(res["filt"], ref["filt"]) <= 1e-10
    assert relerr(res["smo"], ref["smo"]) <= 1e-10
    assert relerr(res["traj"], ref["traj"]) <= 1e-12
    g, gr = res["gradient"], ref["gradient"]
    assert np.max(np.abs(g - gr)) <= 1e-9 * np.max(np.abs(gr)), np.max(np.abs(g - gr), axis=0)
    assert np.array_equal(g == 0.0, gr == 0.0), (np.nonzero(g == 0.0), np.nonzero(gr == 0.0))
    if hessian:
        for k in ("hess1", "hess2"):
            assert np.max(np.abs(res[k] - ref[k])) <= 1e-8 * np.max(np.abs(ref[k])), k


def _ids(runs):
    return ["-".join(str(v) for v in r) for r in runs]


# ------------------------------------------------------------------------------------------------ chain kernel (3)
CHAIN_RUNS = [(lag, m, n) for lag, m in sh.shapes("chain") for n in (5, 37, 1000, 4096)]


@pytest.mark.parametrize("lag,nobs,n", CHAIN_RUNS, ids=_ids(CHAIN_RUNS))
def test_chain_kernel(cuda_dev, lag, nobs, n):
    ref = _oracle(n, nobs, lag, 1)
    _check(_run(cuda_dev, 3, n, nobs, lag, 0, True), ref, CHAIN)
    _check(_run(cuda_dev, 3, n, nobs, lag, 1, True), ref, CHAIN, hessian=True)


# ------------------------------------------------------------------------------------------------ general kernel (1)
GENERAL_N = 3000


@pytest.mark.parametrize("lag,nobs", sh.shapes("general"), ids=_ids(sh.shapes("general")))
def test_general_kernel(cuda_dev, lag, nobs):
    """one CTA and four per problem (another summation order), with and without the Hessian"""
    ref = _oracle(GENERAL_N, nobs, lag, 1)
    for ctas in (1, 4):
        _check(_run(cuda_dev, 1, GENERAL_N, nobs, lag, 0, True, ctas), ref, GENERAL)
        _check(_run(cuda_dev, 1, GENERAL_N, nobs, lag, 1, True, ctas), ref, GENERAL, hessian=True)


# ------------------------------------------------------------------------------------------------ exchange kernel (2)
EXCHANGE_RUNS = [(lag, m, n, c) for lag, m in sh.shapes("exchange") for n, c in ((5000, 5), (65536, 64))]


@pytest.mark.parametrize("lag,nobs,n,ctas", EXCHANGE_RUNS, ids=_ids(EXCHANGE_RUNS))
def test_exchange_kernel(cuda_dev, lag, nobs, n, ctas):
    _check(_run(cuda_dev, 2, n, nobs, lag, 0, True, ctas), _oracle(n, nobs, lag, 0), EXCHANGE)


# ------------------------------------------------------------------------------------------------ grid kernel (6)
GRID_RUNS = [(lag, m, n, c) for lag, m in sh.shapes("grid") for n, c in ((4096, 4), (20000, 0))]


@pytest.mark.parametrize("lag,nobs,n,ctas", GRID_RUNS, ids=_ids(GRID_RUNS))
def test_grid_kernel(cuda_dev, lag, nobs, n, ctas):
    ref = _oracle(n, nobs, lag, 1)
    _check(_run(cuda_dev, 6, n, nobs, lag, 0, True, ctas), ref, GRID)
    _check(_run(cuda_dev, 6, n, nobs, lag, 1, True, ctas), ref, GRID, hessian=True)


# ------------------------------------------------------------------------------------------------ streaming kernels (4, 5)
STREAM_RUNS = [(lag, m, n) for lag, m in sh.shapes("streaming") for n in (3000, 20000)]


@pytest.mark.parametrize("lag,nobs,n", STREAM_RUNS, ids=_ids(STREAM_RUNS))
def test_streaming_kernels(cuda_dev, lag, nobs, n):
    """records (4) and path storage (5), whose jump tables take Q = 0 .. 5 levels over these lags"""
    ref = _oracle(n, nobs, lag, 0)
    for alg in (4, 5):
        _check(_run(cuda_dev, alg, n, nobs, lag, 0, False), ref, STREAMING)


# ------------------------------------------------------------------------------------------------ automatic selection
AUTO_RUNS = [(lag, m, n) for lag, m in ((11, 12), (63, 64), (10, 11)) for n in (1 << 14, 1 << 17)]


@pytest.mark.parametrize("lag,nobs,n", AUTO_RUNS, ids=_ids(AUTO_RUNS))
def test_automatic_selection_where_the_grid_kernel_refuses(cuda_dev, lag, nobs, n):
    """algorithm 0 at N >= 2^14 on shapes outside the grid kernel's rule: status 0 and the oracle's outputs; with the
    Hessian the general kernel (its Hessian compared up to N lag = 2^14 63: the oracle's Hessian branch at 2^17 x 63
    takes minutes)"""
    assert not sh.RULES["grid"](lag, nobs)
    hess_ref = n * lag <= (1 << 14) * 63
    ref = _oracle(n, nobs, lag, int(hess_ref))
    res = _run(cuda_dev, 0, n, nobs, lag, 0, True)
    assert int(res["diag"][DIAG_KERNEL]) in (EXCHANGE, GENERAL), res["diag"]
    _check(res, ref, int(res["diag"][DIAG_KERNEL]))
    _check(_run(cuda_dev, 0, n, nobs, lag, 1, False), ref, GENERAL, hessian=hess_ref)


# ------------------------------------------------------------------------------------------------ rule boundaries
# (algorithm, N, lag, n_obs) one step outside the forced kernel's rule, and that kernel
OUTSIDE = [(3, 1000, 11, 12, CHAIN), (6, 4096, 10, 19, GRID), (6, 4096, 11, 22, GRID), (4, 3000, 10, 19, STREAMING),
           (5, 3000, 63, 125, STREAMING)]


@pytest.mark.parametrize("alg,n,lag,nobs,kernel", OUTSIDE, ids=_ids(OUTSIDE))
def test_forced_kernel_outside_its_rule_runs_another(cuda_dev, alg, n, lag, nobs, kernel):
    """the forced algorithm does not run its kernel one step outside the rule the shape lists assume; the kernel that
    runs instead (the general kernel) matches the oracle"""
    kname = {CHAIN: "chain", GRID: "grid", STREAMING: "streaming"}[kernel]
    assert not sh.RULES[kname](lag, nobs) and sh.entry_accepts(lag, nobs)
    res = _run(cuda_dev, alg, n, nobs, lag, 0, False)
    assert int(res["diag"][DIAG_KERNEL]) not in (kernel, 0), res["diag"]
    _check(res, _oracle(n, nobs, lag, 0), int(res["diag"][DIAG_KERNEL]))


@pytest.mark.parametrize("lag,nobs", [(1, 10), (64, 200), (10, 10), (63, 63)])
def test_entry_refuses_outside_its_region(cuda_dev, lag, nobs):
    from pmmh_qn_b200 import _lib
    from pmmh_qn_b200 import kernels as K
    assert not sh.entry_accepts(lag, nobs)
    obs, params, rvr, _, u = _host(100, nobs, 10)
    with pytest.raises(_lib.PmmhError):
        K.flps_sv_corr(*_dev(cuda_dev, obs, params, rvr, u), lag=lag)


# ------------------------------------------------------------------------------------------------ Philox entry
def test_philox_entry_at_lag_63(cuda_dev):
    """pmmh_flps_sv_corr_philox at lag 63, n_obs = 2 lag: bit for bit the materialised stream on algorithm 5, and the
    oracle on those numbers"""
    import oracle
    import torch
    from pmmh_qn_b200 import kernels as K
    from pmmh_qn_b200.state.particle_methods import split as SP
    n, nobs, lag = 20000, 126, 63
    obs_h = gi.sv_obs(nobs)
    params_h = np.array(gi.SV_PARAM_SETS[1], dtype=np.float64)
    obs, params = _dev(cuda_dev, obs_h, params_h.reshape(1, 4))
    ph = SP.PhiloxRVS(seed=63, offset=126)
    rvr = K.norm_cdf(ph.resampling_normals(nobs, n, cuda_dev))
    a = K.flps_sv_corr_philox(obs, params, rvr, ph.seed, ph.offset, n, lag=lag)
    u = ph.materialise(nobs, n, cuda_dev)
    K.set_sv_algorithm(5)
    try:
        b = K.flps_sv_corr(obs, params, rvr, u, lag=lag)
        torch.cuda.synchronize()
    finally:
        K.set_sv_algorithm(0)
    for k in ("log_like", "filt", "smo", "gradient", "traj", "diag"):
        assert torch.equal(a[k], b[k]), k
    rvp = np.ascontiguousarray(u.cpu().numpy().T).reshape(-1)
    ref = oracle.flps_sv_corr(obs_h, params_h, rvr.cpu().numpy(), rvp, n, lag, 0)
    _check(_np(a), ref, STREAMING)


# ------------------------------------------------------------------------------------------------ host-streamed entry
@pytest.mark.parametrize("nobs", [64, 65])
def test_host_streamed_entry_at_lag_63(cuda_dev, nobs):
    """pmmh_flps_sv_corr_streamed at lag 63 on n_obs = 64 (one 64-step slot of u) and 65 (a second slot of one step):
    bit-identical to the resident entry on the same kernel, and the oracle's outputs"""
    import torch
    from pmmh_qn_b200 import kernels as K
    n, lag = 5000, 63
    rvs = gi.sv_rvs(n, nobs, 600 + nobs)
    obs_h, params_h = gi.sv_obs(nobs), np.array(gi.SV_PARAM_SETS[2], dtype=np.float64)
    rvr_h, rvp = gi.split_particle(rvs, nobs)
    assert K.sv_streamed_eligible(nobs, n, lag)
    obs, params, rvr, u = _dev(cuda_dev, obs_h, params_h.reshape(1, 4), rvr_h, to_time_major(rvp, n, nobs))
    a = K.flps_sv_corr_streamed(rvs, obs, params, rvr, nobs, n, lag=lag)
    torch.cuda.synchronize()
    b = K.flps_sv_corr(obs, params, rvr, u, lag=lag)
    torch.cuda.synchronize()
    assert int(a["diag"][0, DIAG_KERNEL]) == int(b["diag"][0, DIAG_KERNEL])
    for k in ("log_like", "filt", "smo", "gradient", "traj", "diag"):
        assert torch.equal(a[k], b[k]), k
    import oracle
    ref = oracle.flps_sv_corr(obs_h, params_h, rvr_h, rvp, n, lag, 0)
    _check(_np(a), ref, int(a["diag"][0, DIAG_KERNEL]))


# ------------------------------------------------------------------------------------------------ split filter
@pytest.mark.parametrize("world", [1, 2, 3])
def test_split_filter_at_lag_63(cuda_dev, world):
    """LocalComm ranks at lag 63, n_obs = 2 lag (its shortest series): every generation and estimate against the
    oracle"""
    import torch
    from pmmh_qn_b200.state.particle_methods import split as SP
    n, nobs, lag = 5000, 126, 63
    obs, params, rvr, _, u = _host(n, nobs, lag)
    u_d, rvr_d = _dev(cuda_dev, u, rvr)
    out = SP.run_split_smoother(SP.LocalComm(world), obs, params, n, lag, rvr_d, u_d=u_d, device=cuda_dev, cap=n,
                                capc=n, keep_history=True)
    torch.cuda.synchronize()
    ref = _oracle(n, nobs, lag, 0)
    for o in out["per_rank"]:
        assert o["diag"][DIAG_STATUS] == 0, o["diag"]
    for t in range(nobs):
        x = np.concatenate([c.cpu().numpy() for c in out["x_hist"][t]])
        assert relerr(x, ref["X"][t]) <= 1e-12, "generation %d differs from the oracle" % t
    res = {k: out[k].reshape(-1).cpu().numpy() for k in ("filt", "smo", "traj")}
    res["gradient"] = out["gradient"].cpu().numpy().reshape(4, nobs)
    res["log_like"] = float(out["log_like"].item())
    res["diag"] = np.zeros(8, dtype=np.int64)
    _check(res, ref, None)


def test_split_filter_refuses_short_series(cuda_dev):
    """n_obs < 2 lag is refused, not run"""
    from pmmh_qn_b200 import _lib
    from pmmh_qn_b200.state.particle_methods import split as SP
    n, nobs, lag = 5000, 125, 63
    obs, params, rvr, _, u = _host(n, nobs, lag)
    u_d, rvr_d = _dev(cuda_dev, u, rvr)
    with pytest.raises(_lib.PmmhError):
        SP.run_split_smoother(SP.LocalComm(2), obs, params, n, lag, rvr_d, u_d=u_d, device=cuda_dev, cap=n, capc=n)


# ------------------------------------------------------------------------------------------------ model entries
MODEL_SHAPES = [(lag, m) for lag, m in sh.shapes("chain") if m < 2 * lag]
MODEL_N = 1000


def _weights(params, obs, X):
    import generic_pf as gp
    m = gp.SvLeverage(params)
    W = np.zeros_like(X)
    W[0] = 1.0 / X.shape[1]
    for i in range(1, X.shape[0]):
        lw = m.logw(X[i], obs[i])
        sh_ = np.exp(lw - np.max(lw))
        W[i] = sh_ / np.sum(sh_)
    return W


def _check_model8(res, host, n, lag, hess):
    import sv_exact_oracle as so
    obs, params, rvr, rvp = host
    ref = so.flps_sv_exact(params, obs, rvr, rvp, n, lag, dumps=True)
    assert int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
    assert np.array_equal(res["A"][1:], ref["A"][1:])
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"])
    for k in ("filt", "smo"):
        assert relerr(res[k], ref[k]) <= 1e-10, k
    assert relerr(res["traj"], ref["traj"]) <= 1e-12
    X, A = res["X"], res["A"].astype(np.int64)
    r = so.predictive_replay(so.SvLeverageExact(params), obs, X, A, _weights(params, obs, X), lag, hessian=hess)
    g = r[0] if hess else r
    assert np.max(np.abs(res["gradient"] - g)) <= 1e-9 * np.max(np.abs(g))
    assert np.all(res["gradient"][:, -1] == 0.0)
    if hess:
        for got, want in ((res["hess1"], r[1]), (res["hess2"], r[2])):
            assert np.max(np.abs(got - want)) <= 1e-8 * np.max(np.abs(want))


@pytest.mark.parametrize("lag,nobs", MODEL_SHAPES, ids=_ids(MODEL_SHAPES))
def test_model_entry_on_short_series(cuda_dev, lag, nobs):
    """flps_model_corr on the chain kernel at lag + 1 <= n_obs < 2 lag: model 0 bit-identical to the SV entry, model 8
    against its restatement replayed on the kernel's history"""
    from pmmh_qn_b200 import kernels as K
    obs, params, rvr, rvp, u = _host(MODEL_N, nobs, lag)
    d = _dev(cuda_dev, obs, params.reshape(1, 4), rvr, u)
    sv = _run(cuda_dev, 0, MODEL_N, nobs, lag, 0, True)
    m0 = _np(K.flps_model_corr(SV, *d, lag=lag, store_history=True))
    assert int(m0["diag"][DIAG_KERNEL]) == CHAIN == int(sv["diag"][DIAG_KERNEL])
    for k in ("filt", "smo", "log_like", "gradient", "traj", "diag", "X", "A"):
        assert np.array_equal(m0[k], sv[k]), k
    _check(m0, _oracle(MODEL_N, nobs, lag, 0), CHAIN)
    m8 = _np(K.flps_model_corr(SVX, *d, lag=lag, store_history=True))
    assert int(m8["diag"][DIAG_KERNEL]) == CHAIN
    _check_model8(m8, (obs, params, rvr, rvp), MODEL_N, lag, False)


@pytest.mark.parametrize("lag", sh.LAGS["grid"])
def test_model8_hessian_on_the_grid_kernel_at_2lag(cuda_dev, lag):
    """flps_model_batch_corr, model 8 with the Hessian, one problem of 8192 particles at n_obs = 2 lag"""
    from pmmh_qn_b200 import kernels as K
    n, nobs = 8192, 2 * lag
    obs, params, rvr, rvp, u = _host(n, nobs, lag)
    d = _dev(cuda_dev, obs, params.reshape(1, 4), rvr.reshape(1, -1), u[None])
    res = _np(K.flps_model_batch_corr(SVX, *d, lag=lag, compute_hessian=1, store_history=True))
    assert int(res["diag"][DIAG_KERNEL]) == GRID
    _check_model8(res, (obs, params, rvr, rvp), n, lag, True)
