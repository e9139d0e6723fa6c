"""pmmh_filter_model_corr: the particle filter's log-likelihood without the fixed-lag smoother, on the chain kernel
(N <= 4096, any batch, diag kernel 3) and the grid kernel (one problem up to 7168 particles per SM, diag kernel 5).

- On every shape the smoother entry also takes, log_like / filt / traj / diag (and the history X / A) are
  bit-identical to pmmh_flps_model_corr at lag 2 and at lag 10, for the three model ids.
- Series too short for the smoother (n_obs = 2, 3, 5) against the C oracle (SV), oracle/generic_pf.py (linear
  Gaussian, bootstrap and fully adapted) and a one-step NumPy filter built from the generic_pf model callbacks.
- Refusals with their codes (the workspace query refuses the same shapes), workspace sizes, bit reproducibility.
"""
import ctypes

import numpy as np
import pytest

import golden_inputs as gi
from helpers import relerr, to_time_major

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_KERNEL = 2, 6
CHAIN, GRID = 3, 5
TILE_MAX = 7168   # particles of one grid-kernel tile (one CTA per SM)
ERR_INVALID, ERR_WORKSPACE = 1, 2
FILTER_KEYS = ("log_like", "filt", "traj", "diag")


def _dev(cuda_dev, *arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev) for a in arrs]


def _gpu_u(cuda_dev, nobs, n, seed, batch=1):
    """u [batch, nobs, n] (time-major) and rvr [batch, nobs] drawn on the device."""
    import torch
    g = torch.Generator(device=cuda_dev)
    g.manual_seed(seed)
    u = torch.randn((batch, nobs, n), dtype=torch.float64, device=cuda_dev, generator=g)
    rvr = torch.rand((batch, nobs), dtype=torch.float64, device=cuda_dev, generator=g)
    return u, rvr


def _model_inputs(cuda_dev, model_id, nobs, batch):
    """observations shared by the batch and one distinct parameter set per problem"""
    from pmmh_qn_b200 import _lib
    if model_id == _lib.MODEL_SV_LEVERAGE:
        sets, obs = gi.SV_PARAM_SETS, gi.sv_obs(nobs)
    else:
        sets, obs = gi.LG_PARAM_SETS, gi.lg_obs(nobs, gi.LG_PARAM_SETS[0])
    params = np.array([sets[b % len(sets)] for b in range(batch)], dtype=np.float64)
    return _dev(cuda_dev, obs, params)


def _ws_bytes(fn, *args):
    """a workspace query's bytes, or its error code as a negative number"""
    from pmmh_qn_b200 import _lib
    out = ctypes.c_size_t()
    rc = getattr(_lib.load(), fn)(*args, ctypes.byref(out))
    return out.value if rc == 0 else -rc


def _assert_filter_equal(f, s, keys=FILTER_KEYS):
    import torch
    for k in keys:
        assert torch.equal(f[k], s[k]), k


MODELS = [0, 1, 2]


@pytest.mark.parametrize("model_id", MODELS)
@pytest.mark.parametrize("n,batch", [(64, 1), (64, 4), (1000, 1), (1000, 3), (4096, 1), (4096, 3)])
def test_chain_kernel_equals_the_smoother_entry(cuda_dev, model_id, n, batch):
    import torch
    from pmmh_qn_b200 import kernels as K
    nobs = 60
    obs_d, par_d = _model_inputs(cuda_dev, model_id, nobs, batch)
    u, rvr = _gpu_u(cuda_dev, nobs, n, 11 + n + batch, batch)
    f = K.filter_model_corr(model_id, obs_d, par_d, rvr, u)
    torch.cuda.synchronize()
    assert np.all(f["diag"][:, DIAG_KERNEL].cpu().numpy() == CHAIN), f["diag"]
    assert np.all(f["diag"][:, DIAG_STATUS].cpu().numpy() == 0), f["diag"]
    assert "smo" not in f and "gradient" not in f
    for lag in (2, 10):
        s = K.flps_model_corr(model_id, obs_d, par_d, rvr, u, lag=lag)
        torch.cuda.synchronize()
        _assert_filter_equal(f, s)
    if batch > 1:   # the problems of the batch differ
        assert len(set(f["log_like"].cpu().numpy().tolist())) == batch


@pytest.mark.parametrize("model_id", MODELS)
@pytest.mark.parametrize("n", [4097, 1 << 14, 65536, 1 << 20])
def test_grid_kernel_equals_the_smoother_entry(cuda_dev, model_id, n):
    import torch
    from pmmh_qn_b200 import kernels as K
    nobs = 40
    obs_d, par_d = _model_inputs(cuda_dev, model_id, nobs, 1)
    u, rvr = _gpu_u(cuda_dev, nobs, n, 31 + model_id)
    f = K.filter_model_corr(model_id, obs_d, par_d, rvr, u)
    torch.cuda.synchronize()
    assert int(f["diag"][0, DIAG_KERNEL]) == GRID and int(f["diag"][0, DIAG_STATUS]) == 0, f["diag"]
    for lag in (2, 10):
        s = K.flps_model_corr(model_id, obs_d, par_d, rvr, u, lag=lag)
        torch.cuda.synchronize()
        _assert_filter_equal(f, s)


@pytest.mark.parametrize("n,batch", [(1000, 3), (1 << 14, 1)])
def test_history_equals_the_smoother_entry(cuda_dev, n, batch):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    nobs = 30
    obs_d, par_d = _model_inputs(cuda_dev, _lib.MODEL_LINEAR_GAUSSIAN, nobs, batch)
    u, rvr = _gpu_u(cuda_dev, nobs, n, 7, batch)
    f = K.filter_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr, u, store_history=True)
    s = K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr, u, lag=4, store_history=True)
    torch.cuda.synchronize()
    _assert_filter_equal(f, s, FILTER_KEYS + ("X", "A"))
    assert int(f["diag"][0, DIAG_KERNEL]) == (CHAIN if n <= 4096 else GRID)


def _one_step(model, obs, rvr, u1, n):
    """The filter's first step from the generic_pf callbacks: log-likelihood, filt[0..1], traj[0..1]."""
    import generic_pf as gp
    x0 = model.initial_state()
    anc = gp.systematic_corr(np.full(n, 1.0 / n), rvr[1])
    x1 = np.sort(model.propagate(np.full(n, x0)[anc], obs[0], u1), kind="stable")
    lw = model.logw(x1, obs[1])
    mx = np.max(lw)
    sh = np.exp(lw - mx)
    ll = mx + np.log(np.sum(sh)) - np.log(float(n))
    return ll, np.array([x0, np.sum(sh / np.sum(sh) * x1)]), np.array([x0, x1[0]])


@pytest.mark.parametrize("n", [256, 8192])
@pytest.mark.parametrize("nobs", [2, 3, 5])
@pytest.mark.parametrize("model_id", MODELS)
def test_short_series_against_the_oracles(cuda_dev, model_id, nobs, n):
    import generic_pf as gp
    import oracle
    from pmmh_qn_b200 import kernels as K
    if model_id == 0:
        obs, params, rvr, rvp = gi.sv_inputs(n, nobs, 3)
    else:   # model 2 runs on the series as given (they stand for shifted observations), phi < 0
        obs, params, rvr, rvp = gi.lg_inputs(n, nobs, 3 if model_id == 1 else 2)
    callbacks = {0: gp.SvLeverage, 1: gp.LinearGaussian, 2: gp.LinearGaussianFullyAdapted}[model_id]
    obs_d, par_d, rvr_d, u_d = _dev(cuda_dev, obs, params, rvr[:nobs], to_time_major(rvp, n, nobs))
    out = K.filter_model_corr(model_id, obs_d, par_d, rvr_d, u_d)
    res = {k: v[0].cpu().numpy() for k, v in out.items() if not k.startswith("_")}
    assert int(res["diag"][DIAG_KERNEL]) == (CHAIN if n <= 4096 else GRID), res["diag"]
    assert int(res["diag"][DIAG_STATUS]) == 0, res["diag"]
    ll = float(res["log_like"])
    if nobs == 2:
        rll, rfilt, rtraj = _one_step(callbacks(params), obs, rvr, to_time_major(rvp, n, nobs)[1], n)
    else:
        if model_id == 0:
            ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, lag=2)
        else:
            ref = gp.flps_generic(callbacks(params), obs, rvr, rvp, n, lag=2)
        rll, rfilt, rtraj = ref["log_like"], ref["filt"], ref["traj"]
    assert abs(ll - rll) <= 1e-10 * abs(rll), (ll, rll)
    assert relerr(res["filt"], rfilt) <= 1e-10
    assert relerr(res["traj"], rtraj) <= 1e-12


def test_refusals_and_workspace_query(cuda_dev):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    lib = _lib.load()
    sm = K.device_info()[0]
    cap = sm * TILE_MAX

    def call(model_id, nobs, n, batch, hist="both", ws_short=0):
        u, rvr = _gpu_u(cuda_dev, nobs, n, 1, batch)
        obs_d, par_d = _model_inputs(cuda_dev, 1, nobs, batch)
        out = K._sv_outputs(cuda_dev, batch, nobs, n, smoother=False, history=hist != "none")
        xh = out.get("X")
        ah = out.get("A") if hist == "both" else None
        need = _ws_bytes("pmmh_filter_model_workspace_bytes", nobs, n, batch)
        nbytes = max(need, 0) - ws_short
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=cuda_dev)
        rc = lib.pmmh_filter_model_corr(
            model_id, K._ptr(obs_d), 0, K._ptr(par_d), K._ptr(rvr), K._ptr(u), nobs, n, batch, K._ptr(out["filt"]),
            K._ptr(out["log_like"]), K._ptr(out["traj"]), K._ptr(out["diag"]), K._ptr(xh), K._ptr(ah),
            K._ptr(ws), nbytes, K._stream())
        torch.cuda.synchronize()
        return rc

    # shapes: the call and the workspace query refuse them alike
    for nobs, n, batch in [(20, 4097, 2),       # batches of problems above 4096 particles
                           (20, cap + 1, 1),    # above the grid kernel's capacity
                           (20, 1, 1),          # one particle
                           (1, 256, 1),         # one observation
                           (1, 8192, 1)]:
        assert _ws_bytes("pmmh_filter_model_workspace_bytes", nobs, n, batch) == -ERR_INVALID, (nobs, n, batch)
        assert call(1, nobs, n, batch) == ERR_INVALID, (nobs, n, batch)
    # arguments
    assert call(3, 20, 256, 1) == ERR_INVALID                       # unknown model id
    assert call(1, 20, 256, 1, hist="x_only") == ERR_INVALID        # d_x_hist without d_a_hist
    assert call(1, 20, 8192, 1, hist="x_only") == ERR_INVALID
    assert call(1, 20, 8192, 1, ws_short=1) == ERR_WORKSPACE        # one byte short
    # accepted neighbours of the refused shapes
    assert call(1, 20, cap, 1) == 0
    assert call(1, 2, 2, 1) == 0 and call(1, 2, 4097, 1) == 0


def test_workspace_against_the_smoother_entry(cuda_dev):
    from pmmh_qn_b200 import kernels as K
    sm = K.device_info()[0]
    for nobs, n in [(40, 4097), (100, 1 << 14), (300, 65536), (1000, 1 << 20), (1000, sm * TILE_MAX)]:
        f = _ws_bytes("pmmh_filter_model_workspace_bytes", nobs, n, 1)
        s = _ws_bytes("pmmh_flps_model_workspace_bytes", nobs, n, 2, 1)
        assert 0 < f < s, (nobs, n, f, s)
    for nobs, n, batch in [(40, 64, 1), (1000, 4096, 1), (1000, 4096, 1024), (30, 1000, 7)]:
        f = _ws_bytes("pmmh_filter_model_workspace_bytes", nobs, n, batch)
        s = _ws_bytes("pmmh_flps_model_workspace_bytes", nobs, n, 2, batch)
        assert 0 <= f <= s, (nobs, n, batch, f, s)


def test_linear_gaussian_at_2_20_is_bit_reproducible(cuda_dev):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    n, nobs = 1 << 20, 101
    obs_d, par_d = _model_inputs(cuda_dev, _lib.MODEL_LINEAR_GAUSSIAN, nobs, 1)
    u, rvr = _gpu_u(cuda_dev, nobs, n, 9)
    r1 = K.filter_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr, u)
    r2 = K.filter_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, obs_d, par_d, rvr, u)
    torch.cuda.synchronize()
    assert int(r1["diag"][0, DIAG_KERNEL]) == GRID and int(r1["diag"][0, DIAG_STATUS]) == 0
    _assert_filter_equal(r1, r2)
