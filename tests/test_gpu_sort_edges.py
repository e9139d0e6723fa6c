"""The particle sort of every smoother kernel on tied, near-tied and outlying children, up to each kernel's bin capacity.

Inputs come from tests/sort_edge_inputs.py: sibling ties (runs of m children sharing one u), an isolated tie group of
g equal children at generation 1, outliers at +-7, +-12 and +-40 sd (two of them at sorted positions 0 and N - 1),
near-ties a few ulp apart, and a narrow cloud (sigma_v 1e-4, 1e-8).  Every case is compared with the C oracle (SV),
oracle/generic_pf.py (models 1 and 2) or the restatements tests/fa_gradient_oracle.py / fa_hessian_oracle.py (models 4
and 6) at the suite's tolerances: X 1e-12, log-likelihood, filt and smo 1e-10, gradient 1e-9 |g|max, Hessian pieces
1e-8 |H|max.  Ancestors are compared exactly, except under the tie group: its members come from different
equal-valued parents of the one-point generation 0, and the reference's qsort orders them in its own (glibc's) way,
so there the parents' values are compared.  For the same reason the SV Hessian, which reads the flat layout at an
index that depends on the ancestor (quirk Q7), is not run on the tie group.

At sigma_v = 1e-8 exact ties also arise by rounding, between children of different parents of different values.
glibc's merge sort puts such children in descending birth order; every kernel puts them in ascending birth order,
as the NumPy restatement oracle/generic_pf.py does (a stable sort).  The SV cases of that cloud are therefore compared
with the restatement's SV model, ancestors exact, and the SV Hessian (no restatement; quirk Q7) is not run on them.

Capacities (the largest tie group a kernel holds; one more abandons with diag[PMMH_DIAG_STATUS] == 1): chain 1024,
exchange 1024, grid 1024 (a sub-bin), general 4096, streaming 8192.  Under algorithm 0 the general kernel reruns an
abandoned evaluation; the general kernel has no fallback, and the model entries have none at all.
"""
import numpy as np
import pytest

import golden_inputs as gi
import sort_edge_inputs as se
from helpers import first_mismatch_step, relerr

pytestmark = pytest.mark.gpu

DIAG_MAX_BIN, DIAG_STATUS, DIAG_KEY_TIES, DIAG_SOFT_TIES, DIAG_KERNEL = 1, 2, 3, 4, 6
GENERAL, EXCHANGE, CHAIN, STREAMING, GRID = 1, 2, 3, 4, 5
LG, FA, FAG, FAH = 1, 2, 4, 6
LAG = 10
SV = (0.2, 0.9, 0.4, -0.5)

# name -> (builder pattern, builder keywords, sigma_v or None for the default parameters)
CASES = {
    "ties2": ("sibling_ties", dict(m=2), None),
    "ties16": ("sibling_ties", dict(m=16), None),
    "outliers": ("outliers", {}, None),
    "near4": ("near_ties", dict(m=4), None),
    "narrow1e-4": ("plain", {}, 1e-4),
    "narrow1e-8": ("plain", {}, 1e-8),
}
TIED = ("ties2", "ties16")
TIE_FREE = ("outliers", "near4")
# At sigma_v = 1e-8 the children of a step span ~1e9 representable values, so N = 2^14 of them meet exact ties by
# rounding, also between children of different parents (see the module docstring)
ROUNDING_TIES = ("narrow1e-8",)


def _sv_params(case):
    sv = CASES[case][2]
    return np.array(SV if sv is None else (SV[0], SV[1], sv, SV[3]))


def _sv_u(case, n, nobs, seed):
    pattern, kw, _ = CASES[case]
    params = _sv_params(case)
    if pattern == "near_ties":
        kw = dict(kw, sd=se.sv_child_sd(params), xscale=se.sv_xscale(params))
    return se.build(pattern, n, nobs, seed, **kw)


def _rvr(n, nobs, seed):
    return gi.split_particle(gi.sv_rvs(n, nobs, seed), nobs)[0]


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def _np(out, b=0):
    return {k: v[b].cpu().numpy() for k, v in out.items() if not k.startswith("_")}


def _with_algorithm(alg, fn):
    from pmmh_qn_b200 import kernels as K
    K.set_sv_algorithm(alg)
    try:
        return fn()
    finally:
        K.set_sv_algorithm(0)


def _check_ancestors(res, ref, by_value=False, grid=False):
    """ancestors exact (by_value: the parents' values); True if the outputs can be compared in full.  On the grid
    kernel a first differing generation may come with a counted soft tie (as in test_gpu_shift_edges.py): the
    generations before it must agree, and the outputs are then not compared."""
    A, Ar, Xr = res["A"].astype(np.int64), ref["A"].astype(np.int64), ref["X"]
    if by_value:
        for t in range(1, A.shape[0]):
            assert np.array_equal(Xr[t - 1][A[t]], Xr[t - 1][Ar[t]]), "parent values differ at time %d" % t
        return True
    step = first_mismatch_step(A[1:], Ar[1:])
    if step is None:
        return True
    assert grid and int(res["diag"][DIAG_SOFT_TIES]) > 0, "ancestors differ first at time %d" % (step + 1)
    assert relerr(res["X"][:step + 1], Xr[:step + 1]) <= 1e-12
    return False


def _check(res, ref, by_value=False, grid=False, hessian=False, zero_gradient=False):
    """one problem's outputs (NumPy) against the reference"""
    assert int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
    if "A" in res and not _check_ancestors(res, ref, by_value, grid):
        return
    if "X" in res:
        assert relerr(res["X"], ref["X"]) <= 1e-12
    assert np.isfinite(ref["log_like"])
    assert abs(float(res["log_like"]) - ref["log_like"]) <= 1e-10 * abs(ref["log_like"]), (res["log_like"],
                                                                                            ref["log_like"])
    assert relerr(res["filt"], ref["filt"]) <= 1e-10
    if "smo" in ref:
        assert relerr(res["smo"], ref["smo"]) <= 1e-10
    assert relerr(res["traj"], ref["traj"]) <= 1e-12
    if "gradient" in ref:
        g = res["gradient"]
        if zero_gradient:
            assert np.all(g == 0.0)
        else:
            assert np.max(np.abs(g - ref["gradient"])) <= 1e-9 * np.max(np.abs(ref["gradient"]))
    if hessian:
        for k in ("hess1", "hess2"):
            assert np.max(np.abs(res[k] - ref[k])) <= 1e-8 * np.max(np.abs(ref[k])), k


def _check_ties_counted(res, case):
    ties = int(res["diag"][DIAG_KEY_TIES])
    if case in TIED:
        assert ties > 0, res["diag"]
    elif case in TIE_FREE:
        assert ties == 0, res["diag"]


# ------------------------------------------------------------------------------------------------ SV entry
# algorithm -> (N, kernel it runs, history output, Hessian runs)
SV_ALGS = {
    1: (5000, GENERAL, True, True),
    2: (5000, EXCHANGE, True, False),
    3: (1000, CHAIN, True, True),
    4: (5000, STREAMING, False, False),
    5: (5000, STREAMING, False, False),
    6: (5000, GRID, True, True),
    0: (1 << 14, GRID, True, True),
}
SV_RUNS = [(a, c, h) for a in SV_ALGS for c in CASES
           for h in ((0, 1) if SV_ALGS[a][3] and c not in ROUNDING_TIES else (0,))]


def _sv_reference(case, obs, params, rvr, rvp, n, hess):
    """the C oracle, or for a cloud with rounding ties the restatement, whose stable sort orders equal children of
    different parents by birth row as the kernels do"""
    import generic_pf as gp
    import oracle
    if case in ROUNDING_TIES:
        assert not hess
        return gp.flps_generic(gp.SvLeverage(params), obs, rvr, rvp, n, LAG, dumps=True)
    return oracle.flps_sv_corr(obs, params, rvr, rvp, n, LAG, hess, dumps=True)


def _sv_run(cuda_dev, alg, obs, params, rvr, u, hess=0, hist=True):
    import torch
    from pmmh_qn_b200 import kernels as K
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, params, rvr, u)

    def run():
        out = K.flps_sv_corr(obs_d, par_d, rvr_d, u_d, lag=LAG, compute_hessian=hess, store_history=hist)
        torch.cuda.synchronize()
        return out
    return _np(_with_algorithm(alg, run))


@pytest.mark.parametrize("alg,case,hess", SV_RUNS, ids=["a%d-%s-h%d" % r for r in SV_RUNS])
def test_sv_entry_vs_oracle(cuda_dev, alg, case, hess):
    """algorithms 1 .. 6 alone and 0 (grid kernel, with its fallback pass) on sibling ties, outliers, near-ties
    and narrow clouds: no kernel abandons, every output matches the oracle, and equal keys are counted exactly
    when there are ties"""
    n, kernel, hist, _ = SV_ALGS[alg]
    nobs = 40
    params = _sv_params(case)
    u, rvp = _sv_u(case, n, nobs, 11 + alg)
    obs, rvr = gi.sv_obs(nobs), _rvr(n, nobs, 11 + alg)
    ref = _sv_reference(case, obs, params, rvr, rvp, n, hess)
    res = _sv_run(cuda_dev, alg, obs, params, rvr, u, hess, hist)
    assert int(res["diag"][DIAG_KERNEL]) == kernel, res["diag"]
    _check(res, ref, grid=kernel == GRID, hessian=bool(hess))
    _check_ties_counted(res, case)


# kernel -> (algorithm run alone, N, largest tie group it holds, fallback under algorithm 0: None, "oracle" (the
# chain kernel's fallback runs the general kernel on one CTA: another summation order) or "bitwise" (the same
# general kernel launch as algorithm 1))
CAPACITY = {
    "chain": (3, 4096, 1024, CHAIN, "oracle"),
    "exchange": (2, 8192, 1024, EXCHANGE, "bitwise"),
    "grid": (6, 1 << 14, 1024, GRID, "bitwise"),
    "general": (1, 12000, 4096, GENERAL, None),
    "streaming": (5, 20000, 8192, STREAMING, None),
}
CAP_RUNS = [(k, o) for k in CAPACITY for o in (0, 1)]
CAP_NOBS = 24


def _group(n, g, seed):
    return se.build("tie_group", n, CAP_NOBS, seed, g=g)


@pytest.mark.parametrize("kernel,over", CAP_RUNS, ids=["%s-cap+%d" % r for r in CAP_RUNS])
def test_sv_tie_group_at_capacity(cuda_dev, kernel, over):
    """a tie group of the capacity holds and matches the oracle; one more abandons the kernel run alone, and
    algorithm 0's fallback pass gives the oracle's outputs (bit-identical to algorithm 1 where it is the same
    general-kernel launch)"""
    import oracle
    alg, n, cap, kid, fallback = CAPACITY[kernel]
    g = cap + over
    hist = kid != STREAMING
    u, rvp = _group(n, g, 21 + over)
    obs, params, rvr = gi.sv_obs(CAP_NOBS), np.array(SV), _rvr(n, CAP_NOBS, 21)
    ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, LAG, 0, dumps=True)
    res = _sv_run(cuda_dev, alg, obs, params, rvr, u, 0, hist)
    assert int(res["diag"][DIAG_KERNEL]) == kid, res["diag"]
    if over == 0:
        _check(res, ref, by_value=True, grid=kid == GRID)
        assert int(res["diag"][DIAG_MAX_BIN]) >= g, res["diag"]
        assert int(res["diag"][DIAG_KEY_TIES]) > 0, res["diag"]
    else:
        assert int(res["diag"][DIAG_STATUS]) == 1, "%s kernel held a tie group of %d: %s" % (kernel, g, res["diag"])
    if fallback is None:
        return
    auto = _sv_run(cuda_dev, 0, obs, params, rvr, u, 0, hist)
    assert int(auto["diag"][DIAG_KERNEL]) == (kid if over == 0 else GENERAL), auto["diag"]
    _check(auto, ref, by_value=True, grid=kid == GRID and over == 0)
    if over == 1 and fallback == "bitwise":
        one = _sv_run(cuda_dev, 1, obs, params, rvr, u, 0, hist)
        for k in ("filt", "smo", "log_like", "gradient", "traj", "X", "A"):
            assert np.array_equal(auto[k], one[k]), k


def test_general_kernel_beyond_its_bin_capacity(cuda_dev):
    """a tie group above kBinCap = 4096: the general kernel (the last kernel, also under algorithm 0) abandons
    with a NaN log-likelihood, and the estimator reports the failed evaluation"""
    from pmmh_qn_b200 import ParticleMethodsCUDA
    from toy_models import ToySVModel
    n, g = 12000, 4097
    u, rvp = _group(n, g, 31)
    obs, params = gi.sv_obs(CAP_NOBS), np.array(SV)
    raw = gi.sv_rvs(n, CAP_NOBS, 31).reshape(-1)[:CAP_NOBS]
    rvr = gi.split_particle(raw, CAP_NOBS)[0]
    for alg in (1, 0):
        res = _sv_run(cuda_dev, alg, obs, params, rvr, u, 0, False)
        assert int(res["diag"][DIAG_KERNEL]) == GENERAL and int(res["diag"][DIAG_STATUS]) == 1, res["diag"]
        assert np.isnan(res["log_like"])
    model = ToySVModel(obs, params)
    est = ParticleMethodsCUDA(model, no_particles=n, fixed_lag=LAG)
    rvs = np.concatenate([raw, rvp]).reshape(CAP_NOBS, n + 1)
    assert est.smoother(model, rvs={'rvs': rvs}) is False
    assert est.diagnostics["status"] == 1


# ------------------------------------------------------------------------------------------------ bootstrap filter
@pytest.mark.parametrize("case", ["ties2", "ties16", "outliers", "near4"])
def test_bpf_vs_oracle(cuda_dev, case):
    import oracle
    import torch
    from pmmh_qn_b200 import kernels as K
    n, nobs = 5000, 40
    u, rvp = _sv_u(case, n, nobs, 41)
    obs, params, rvr = gi.sv_obs(nobs), _sv_params(case), _rvr(n, nobs, 41)
    ref = oracle.bpf_sv_corr(obs, params, rvr, rvp, n, dumps=True)
    out = K.bpf_sv_corr(*_dev(cuda_dev, obs, params, rvr, u), store_history=True)
    torch.cuda.synchronize()
    res = _np(out)
    assert int(res["diag"][DIAG_KERNEL]) == GENERAL, res["diag"]
    _check(res, ref)


# ------------------------------------------------------------------------------------------------ model entries
def _model_inputs(model_id, case, n, nobs, seed, g=None):
    """(obs, params, rvr, u, rvp, reference) of a linear Gaussian model; the fully adapted models take the shifted
    series"""
    import fa_gradient_oracle as fo
    import generic_pf as gp
    params = np.array(gi.LG_PARAM_SETS[0])
    if case in CASES and CASES[case][2] is not None:
        params[1] = CASES[case][2]
    if g is not None:
        u, rvp = se.build("tie_group", n, nobs, seed, g=g)
    elif case == "plain":
        u, rvp = se.build("plain", n, nobs, seed)
    else:
        pattern, kw, _ = CASES[case]
        if pattern == "near_ties":
            kw = dict(kw, sd=params[1], xscale=8.0)
        u, rvp = se.build(pattern, n, nobs, seed, **kw)
    full = gi.lg_obs(nobs + 1, gi.LG_PARAM_SETS[0])
    obs = full[:nobs] if model_id == LG else full[1:]
    rvr = _rvr(n, nobs, seed)
    if model_id == LG:
        ref = gp.flps_generic(gp.LinearGaussian(params), obs, rvr, rvp, n, LAG, dumps=True)
    elif model_id == FA:
        ref = gp.flps_generic(gp.LinearGaussianFullyAdapted(params), obs, rvr, rvp, n, LAG, dumps=True)
    else:
        ref = fo.flps_fa_grad(params, obs, rvr, rvp, n, LAG, dumps=True)
    return obs, params, rvr, u, rvp, ref


MODEL_RUNS = [(m, k, c) for m in (LG, FA, FAG) for k in (CHAIN, GRID) for c in CASES]


@pytest.mark.parametrize("model_id,kernel,case", MODEL_RUNS, ids=["m%d-k%d-%s" % r for r in MODEL_RUNS])
def test_model_entry_vs_reference(cuda_dev, model_id, kernel, case):
    """flps_model_corr for models 1, 2 and 4 on the chain (N = 1000) and grid (N = 5000) kernels; the filter entry
    gives the smoother's filt, log-likelihood and trajectory bit for bit"""
    from pmmh_qn_b200 import kernels as K
    n, nobs = (1000 if kernel == CHAIN else 5000), 40
    obs, params, rvr, u, _, ref = _model_inputs(model_id, case, n, nobs, 50 + model_id)
    d = _dev(cuda_dev, obs, params, rvr, u)
    res = _np(K.flps_model_corr(model_id, *d, lag=LAG, store_history=True))
    assert int(res["diag"][DIAG_KERNEL]) == kernel, res["diag"]
    _check(res, ref, grid=kernel == GRID, zero_gradient=model_id == FA)
    _check_ties_counted(res, case)
    filt = _np(K.filter_model_corr(model_id, *d, store_history=True))
    for k in ("filt", "log_like", "traj", "X", "A"):
        assert np.array_equal(filt[k], res[k]), k


MODEL_CAP_RUNS = [(m, k, o) for m in (LG, FAG) for k in (CHAIN, GRID) for o in (0, 1)]


@pytest.mark.parametrize("model_id,kernel,over", MODEL_CAP_RUNS, ids=["m%d-k%d-cap+%d" % r for r in MODEL_CAP_RUNS])
def test_model_entry_tie_group_at_capacity(cuda_dev, model_id, kernel, over):
    """a tie group of 1024 holds on the chain (N = 4096) and grid (N = 2^14) kernels; 1025 reports status 1 (the
    model entries have no fallback pass) and the estimator reports the failed evaluation"""
    from pmmh_qn_b200 import kernels as K
    n, g = (4096 if kernel == CHAIN else 1 << 14), 1024 + over
    obs, params, rvr, u, rvp, ref = _model_inputs(model_id, None, n, CAP_NOBS, 60 + over, g=g)
    res = _np(K.flps_model_corr(model_id, *_dev(cuda_dev, obs, params, rvr, u), lag=LAG, store_history=True))
    assert int(res["diag"][DIAG_KERNEL]) == kernel, res["diag"]
    if over == 0:
        _check(res, ref, by_value=True, grid=kernel == GRID)
        assert int(res["diag"][DIAG_MAX_BIN]) >= g and int(res["diag"][DIAG_KEY_TIES]) > 0, res["diag"]
        return
    assert int(res["diag"][DIAG_STATUS]) == 1, res["diag"]
    if model_id == FAG:
        from pmmh_qn_b200 import LinearGaussianParticleMethodsCUDA
        from test_gpu_fa_gradient_kalman import ToyLGSSModel
        model = ToyLGSSModel(gi.lg_obs(CAP_NOBS + 1, gi.LG_PARAM_SETS[0]), params)
        est = LinearGaussianParticleMethodsCUDA(model, n, fixed_lag=LAG)
        raw = gi.sv_rvs(n, CAP_NOBS, 60 + over).reshape(-1)[:CAP_NOBS]
        rvs = np.concatenate([raw, rvp]).reshape(CAP_NOBS, n + 1)
        assert est.smoother(model, rvs={'rvs': rvs}) is False
        assert est.diagnostics["status"] == 1


def _fa_weights(params, obs, X):
    import generic_pf as gp
    m = gp.LinearGaussianFullyAdapted(params)
    W = np.zeros_like(X)
    W[0] = 1.0 / X.shape[1]
    for i in range(1, X.shape[0]):
        lw = m.logw(X[i], obs[i])
        sh = np.exp(lw - np.max(lw))
        W[i] = sh / np.sum(sh)
    return W


def _check_fa_hessian(res, params, obs):
    import fa_hessian_oracle as fh
    X, A = res["X"], res["A"].astype(np.int64)
    h1, h2 = fh.predictive_hessian(fh.LinearGaussianFullyAdaptedHess(params), obs, X, A, _fa_weights(params, obs, X),
                                   LAG)
    for got, want in ((res["hess1"], h1), (res["hess2"], h2)):
        assert np.max(np.abs(got - want)) <= 1e-8 * np.max(np.abs(want)), (got, want)


@pytest.mark.parametrize("case", ["ties2", "ties16", "outliers", "near4", "narrow1e-4", "group1024"])
def test_model6_hessian_on_the_grid_kernel(cuda_dev, case):
    """model 6's hess1 / hess2 against the restatement replayed on the kernel's own history (so the order of a tie
    group cannot matter); the other outputs against model 4's reference"""
    from pmmh_qn_b200 import kernels as K
    n, nobs = 1 << 14, 32
    g = 1024 if case == "group1024" else None
    obs, params, rvr, u, _, ref = _model_inputs(FAG, None if g else case, n, nobs, 70, g=g)
    par = np.asarray(params).reshape(1, 4)
    res = _np(K.flps_model_batch_corr(FAH, *_dev(cuda_dev, obs, par, rvr, u), lag=LAG, compute_hessian=1,
                                      store_history=True))
    assert int(res["diag"][DIAG_KERNEL]) == GRID, res["diag"]
    _check(res, ref, by_value=g is not None, grid=True)
    _check_fa_hessian(res, params, obs)


# ------------------------------------------------------------------------------------------------ team batches
BATCH, BATCH_N, BATCH_NOBS = 20, 1 << 14, 24
BATCH_RUNS = [(m, a) for m in (0, FAH) for a in ("ties16", "group1025")]


@pytest.mark.parametrize("model_id,adv", BATCH_RUNS, ids=["m%d-%s" % r for r in BATCH_RUNS])
def test_team_batch_with_adversarial_problems(cuda_dev, model_id, adv):
    """flps_model_batch_corr with the Hessian (SV and model 6), 20 problems of 2^14 particles (more than one wave of
    teams): the first and the last problem are adversarial, and every other problem is bit-identical to its
    one-problem run; an adversarial problem matches its reference, or reports status 1 at capacity + 1"""
    import oracle
    import torch
    from pmmh_qn_b200 import kernels as K
    n, nobs = BATCH_N, BATCH_NOBS
    adversarial = (0, BATCH - 1)
    probs = []
    for b in range(BATCH):
        seed = 80 + b
        if model_id == 0:
            obs, params, rvr = gi.sv_obs(nobs), np.array(SV), _rvr(n, nobs, seed)
            if b in adversarial:
                u, rvp = (_sv_u(adv, n, nobs, seed) if adv != "group1025" else _group(n, 1025, seed))
            else:
                u, rvp = se.build("plain", n, nobs, seed)
            probs.append((obs, params, rvr, u, rvp))
        else:
            g = 1025 if (b in adversarial and adv == "group1025") else None
            case = adv if b in adversarial else "plain"
            obs, params, rvr, u, rvp, _ = _model_inputs(FAG, None if g else case, n, nobs, seed, g=g)
            probs.append((obs, params, rvr, u, rvp))
    obs_d, par_d, rvr_d, u_d = (torch.stack(_dev(cuda_dev, *[p[i] for p in probs])) for i in range(4))
    out = K.flps_model_batch_corr(model_id, obs_d, par_d, rvr_d, u_d, lag=LAG, compute_hessian=1, store_history=True)
    torch.cuda.synchronize()
    for b in range(BATCH):
        res = _np(out, b)
        assert int(res["diag"][DIAG_KERNEL]) == GRID, (b, res["diag"])
        obs, params, rvr, u, rvp = probs[b]
        if b not in adversarial:
            one = _np(K.flps_model_batch_corr(model_id, *_dev(cuda_dev, obs[None], params[None], rvr[None], u[None]),
                                              lag=LAG, compute_hessian=1, store_history=True))
            for k in ("filt", "smo", "log_like", "gradient", "traj", "hess1", "hess2", "diag", "X", "A"):
                assert np.array_equal(res[k], one[k]), (b, k)
            continue
        if adv == "group1025":
            assert int(res["diag"][DIAG_STATUS]) == 1, (b, res["diag"])
            continue
        if model_id == 0:
            ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, LAG, 1, dumps=True)
            _check(res, ref, grid=True, hessian=True)
        else:
            assert int(res["diag"][DIAG_STATUS]) == 0, (b, res["diag"])
            _check_fa_hessian(res, params, obs)


# ------------------------------------------------------------------------------------------------ split filter
def _split(cuda_dev, world, obs, params, rvr, u, n):
    import torch
    from pmmh_qn_b200.state.particle_methods import split as SP
    u_d, rvr_d = _dev(cuda_dev, u, rvr)
    out = SP.run_split_smoother(SP.LocalComm(world), obs, params, n, LAG, rvr_d, u_d=u_d, device=cuda_dev, cap=n,
                                capc=n, keep_history=True)
    torch.cuda.synchronize()
    return out


def _check_split(out, ref):
    for o in out["per_rank"]:
        assert o["diag"][DIAG_STATUS] == 0, o["diag"]
    for t in range(ref["X"].shape[0]):
        x = np.concatenate([c.cpu().numpy() for c in out["x_hist"][t]])
        assert relerr(x, ref["X"][t]) <= 1e-12, "generation %d differs from the oracle" % t
    res = {k: out[k].reshape(-1).cpu().numpy() if k != "gradient" else out[k].cpu().numpy()
           for k in ("filt", "smo", "traj", "gradient")}
    res["log_like"] = float(out["log_like"].item())
    res["diag"] = np.zeros(8, dtype=np.int64)
    _check(res, ref)


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("case", ["ties16", "outliers"])
def test_split_filter_vs_oracle(cuda_dev, case, world):
    import oracle
    n, nobs = 5000, 40
    u, rvp = _sv_u(case, n, nobs, 90)
    obs, params, rvr = gi.sv_obs(nobs), _sv_params(case), _rvr(n, nobs, 90)
    ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, LAG, 0, dumps=True)
    _check_split(_split(cuda_dev, world, obs, params, rvr, u, n), ref)


@pytest.mark.parametrize("over", [0, 1])
def test_split_filter_tie_group_at_capacity(cuda_dev, over):
    """a tie group of kMaxBinRank = 8192 holds; 8193 abandons with the FloatingPointError split.py documents"""
    import oracle
    n, g = 20000, 8192 + over
    u, rvp = _group(n, g, 95)
    obs, params, rvr = gi.sv_obs(CAP_NOBS), np.array(SV), _rvr(n, CAP_NOBS, 95)
    if over:
        with pytest.raises(FloatingPointError):
            _split(cuda_dev, 2, obs, params, rvr, u, n)
        return
    ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, LAG, 0, dumps=True)
    _check_split(_split(cuda_dev, 2, obs, params, rvr, u, n), ref)
