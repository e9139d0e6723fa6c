"""pmmh_flps_model_batch_corr / pmmh_filter_model_batch_corr: batches on the grid kernel (csrc/sv_grid.cu), one team
of ceil(N / 2048) CTAs per problem, in waves of floor(SMs / G) teams.  The teams use the one-problem tiles, so every
output of problem b must equal the one-problem grid run on that problem bit for bit:

- smoother, models 0 / 1 / 2, distinct parameters, observations and u per problem: N = 4097 (G = 3), N = 2^14 with B
  below, equal to and above the team count (partial last wave), N = 2^16 with B = 3, 4, 9, N = 2^18 with B = 2
  (one team per wave), N = 2^20 with B = 2;
- the SV Hessian against pmmh_flps_sv_corr on the grid kernel (algorithm 6);
- the filter entry against pmmh_filter_model_corr and the smoother batch entry; history over several waves;
- a degenerate problem (u = 0) is abandoned alone, in the first and in the last wave;
- refusals and workspace size; a full wave run twice.
Team counts are derived from the device's SM count.
"""
import ctypes

import numpy as np
import pytest

import golden_inputs as gi

pytestmark = pytest.mark.gpu

DIAG_STATUS, DIAG_KERNEL, DIAG_COUNT = 2, 6, 8
GRID = 5
SMO_KEYS = ("log_like", "filt", "smo", "gradient", "traj", "diag")
FILTER_KEYS = ("log_like", "filt", "traj", "diag")


def _teams(n, batch=1 << 30):
    from pmmh_qn_b200 import kernels as K
    sm = K.device_info()[0]
    G = min(max((n + 2047) // 2048, 1), sm)
    return max(1, min(batch, sm // G))


def _inputs(cuda_dev, model, n, nobs, batch, seed, per_problem_obs=True):
    """obs ([B, nobs] or shared [nobs]), params [B, 4], rvr [B, nobs], u [B, nobs, n]: distinct per problem"""
    import torch
    sets = gi.SV_PARAM_SETS if model == 0 else gi.LG_PARAM_SETS
    params = np.array([sets[(seed + b) % len(sets)] for b in range(batch)], dtype=np.float64)
    params[:, 1] *= 1.0 - 0.01 * (np.arange(batch) % 7)   # phi: no two problems alike
    if model == 0:
        obs = np.stack([gi.sv_obs(nobs, seed=100 + seed + b) for b in range(batch)])
    else:
        obs = np.stack([gi.lg_obs(nobs, tuple(params[b]), seed=200 + seed + b) for b in range(batch)])
    if not per_problem_obs:
        obs = obs[0]
    g = torch.Generator(device=cuda_dev)
    g.manual_seed(seed)
    u = torch.randn((batch, nobs, n), dtype=torch.float64, device=cuda_dev, generator=g)
    rvr = torch.rand((batch, nobs), dtype=torch.float64, device=cuda_dev, generator=g)
    obs_d = torch.from_numpy(np.ascontiguousarray(obs)).to(cuda_dev)
    par_d = torch.from_numpy(params).to(cuda_dev)
    return obs_d, par_d, rvr, u


def _obs_of(obs, b):
    return obs if obs.dim() == 1 else obs[b:b + 1].contiguous()


def _single(model, obs, params, rvr, u, b, lag, hess=False, history=False):
    """the one-problem grid run on problem b"""
    from pmmh_qn_b200 import kernels as K
    args = (_obs_of(obs, b), params[b:b + 1].contiguous(), rvr[b:b + 1].contiguous(), u[b:b + 1].contiguous())
    if hess:
        K.set_sv_algorithm(6)
        try:
            return K.flps_sv_corr(*args, lag=lag, compute_hessian=True, store_history=history)
        finally:
            K.set_sv_algorithm(0)
    return K.flps_model_corr(model, *args, lag=lag, store_history=history)


def _assert_same(batch_out, single_out, b, keys):
    import torch
    for k in keys:
        assert torch.equal(batch_out[k][b], single_out[k][0]), (k, b)


def _assert_batch_equals_singles(model, n, nobs, batch, lag, seed, cuda_dev, per_problem_obs=True):
    import torch
    from pmmh_qn_b200 import kernels as K
    obs, params, rvr, u = _inputs(cuda_dev, model, n, nobs, batch, seed, per_problem_obs)
    out = K.flps_model_batch_corr(model, obs, params, rvr, u, lag=lag)
    torch.cuda.synchronize()
    d = out["diag"].cpu().numpy()
    assert np.all(d[:, DIAG_KERNEL] == GRID) and np.all(d[:, DIAG_STATUS] == 0), d
    for b in range(batch):
        ref = _single(model, obs, params, rvr, u, b, lag)
        torch.cuda.synchronize()
        _assert_same(out, ref, b, SMO_KEYS)


@pytest.mark.parametrize("model", [0, 1, 2])
def test_batch_4097_three_ctas_per_team(cuda_dev, model):
    _assert_batch_equals_singles(model, 4097, 50, 5, 10, 1, cuda_dev)


@pytest.mark.parametrize("model", [0, 1, 2])
@pytest.mark.parametrize("which", ["below", "equal", "above"])
def test_batch_2_14_around_the_team_count(cuda_dev, model, which):
    nt = _teams(1 << 14)
    batch = {"below": max(1, nt // 3), "equal": nt, "above": nt + nt // 2 + 1}[which]
    _assert_batch_equals_singles(model, 1 << 14, 44, batch, 10, 2 + model, cuda_dev, per_problem_obs=model != 1)


@pytest.mark.parametrize("model", [0, 1, 2])
@pytest.mark.parametrize("batch", [3, 4, 9])
def test_batch_2_16(cuda_dev, model, batch):
    _assert_batch_equals_singles(model, 1 << 16, 40, batch, 4, 3, cuda_dev)


@pytest.mark.parametrize("model", [0, 1, 2])
def test_batch_2_18_one_team_per_wave(cuda_dev, model):
    _assert_batch_equals_singles(model, 1 << 18, 40, 2, 10, 4, cuda_dev)


def test_batch_2_20_T300(cuda_dev):
    _assert_batch_equals_singles(1, 1 << 20, 301, 2, 10, 5, cuda_dev)


@pytest.mark.parametrize("n,batch", [(1 << 14, 20), (1 << 16, 5)])
def test_sv_hessian_batch_equals_grid_runs(cuda_dev, n, batch):
    import torch
    from pmmh_qn_b200 import kernels as K
    obs, params, rvr, u = _inputs(cuda_dev, 0, n, 50, batch, 6)
    out = K.flps_model_batch_corr(0, obs, params, rvr, u, lag=10, compute_hessian=1)
    torch.cuda.synchronize()
    assert np.all(out["diag"][:, DIAG_STATUS].cpu().numpy() == 0)
    for b in range(batch):
        ref = _single(0, obs, params, rvr, u, b, 10, hess=True)
        torch.cuda.synchronize()
        assert int(ref["diag"][0, DIAG_KERNEL]) == GRID
        _assert_same(out, ref, b, SMO_KEYS + ("hess1", "hess2"))


@pytest.mark.parametrize("model", [0, 1, 2])
def test_filter_batch_equals_filter_runs_and_smoother_batch(cuda_dev, model):
    import torch
    from pmmh_qn_b200 import kernels as K
    n = 1 << 14
    batch = _teams(n) + 3
    obs, params, rvr, u = _inputs(cuda_dev, model, n, 45, batch, 7)
    f = K.filter_model_batch_corr(model, obs, params, rvr, u)
    s = K.flps_model_batch_corr(model, obs, params, rvr, u, lag=10)
    torch.cuda.synchronize()
    for k in FILTER_KEYS:
        assert torch.equal(f[k], s[k]), k
    for b in range(batch):
        ref = K.filter_model_corr(model, _obs_of(obs, b), params[b:b + 1].contiguous(), rvr[b:b + 1].contiguous(),
                                  u[b:b + 1].contiguous())
        torch.cuda.synchronize()
        _assert_same(f, ref, b, FILTER_KEYS)


def test_history_over_several_waves(cuda_dev):
    import torch
    from pmmh_qn_b200 import kernels as K
    n = 1 << 16
    batch = 2 * _teams(n) + 1
    obs, params, rvr, u = _inputs(cuda_dev, 1, n, 40, batch, 8)
    out = K.flps_model_batch_corr(1, obs, params, rvr, u, lag=10, store_history=True)
    fo = K.filter_model_batch_corr(1, obs, params, rvr, u, store_history=True)
    torch.cuda.synchronize()
    for b in range(batch):
        ref = _single(1, obs, params, rvr, u, b, 10, history=True)
        torch.cuda.synchronize()
        _assert_same(out, ref, b, SMO_KEYS + ("X", "A"))
        _assert_same(fo, ref, b, ("X", "A"))


@pytest.mark.parametrize("where", ["first", "last"])
def test_abandoned_problem_leaves_the_others_alone(cuda_dev, where):
    import torch
    from pmmh_qn_b200 import kernels as K
    n = 1 << 14
    batch = _teams(n) + 3   # two waves
    obs, params, rvr, u = _inputs(cuda_dev, 0, n, 40, batch, 9)
    bad = 0 if where == "first" else batch - 1
    u[bad].zero_()   # degenerate cloud: every child of a parent has the parent's propagated value
    out = K.flps_model_batch_corr(0, obs, params, rvr, u, lag=10)
    torch.cuda.synchronize()
    st = out["diag"][:, DIAG_STATUS].cpu().numpy()
    assert st[bad] == 1 and np.all(np.delete(st, bad) == 0), st
    for b in range(batch):
        if b == bad:
            continue
        ref = _single(0, obs, params, rvr, u, b, 10)
        torch.cuda.synchronize()
        _assert_same(out, ref, b, SMO_KEYS)


def test_full_wave_is_bit_reproducible(cuda_dev):
    import torch
    from pmmh_qn_b200 import kernels as K
    n = 1 << 14
    batch = _teams(n)
    obs, params, rvr, u = _inputs(cuda_dev, 0, n, 60, batch, 10)
    ws = K.Workspace()
    r1 = K.flps_model_batch_corr(0, obs, params, rvr, u, lag=10, workspace=ws)
    r2 = K.flps_model_batch_corr(0, obs, params, rvr, u, lag=10, workspace=ws)
    torch.cuda.synchronize()
    for k in SMO_KEYS:
        assert torch.equal(r1[k], r2[k]), k


def _flps_ws(nobs, n, lag, batch, hess=0):
    from pmmh_qn_b200 import _lib
    out = ctypes.c_size_t()
    rc = _lib.load().pmmh_flps_model_batch_workspace_bytes(nobs, n, lag, batch, hess, ctypes.byref(out))
    return out.value if rc == 0 else None


def _filter_ws(nobs, n, batch):
    from pmmh_qn_b200 import _lib
    out = ctypes.c_size_t()
    rc = _lib.load().pmmh_filter_model_batch_workspace_bytes(nobs, n, batch, ctypes.byref(out))
    return out.value if rc == 0 else None


def test_refusals_and_workspace(cuda_dev):
    import torch
    from pmmh_qn_b200 import _lib, kernels as K
    lib = _lib.load()
    sm = K.device_info()[0]

    def call(model, n, nobs, lag, batch, hess=0, x_only=False, ws_bytes=None):
        """pmmh_flps_model_batch_corr's status on small buffers (the refusals come before any launch)"""
        obs, params, rvr, u = _inputs(cuda_dev, 0, n, nobs, batch, 11)
        f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device=cuda_dev)   # noqa: E731
        filt, smo, traj, ll, grad = f64(batch, nobs), f64(batch, nobs), f64(batch, nobs), f64(batch), f64(batch, 4, nobs)
        h1, h2 = f64(batch, 16), f64(batch, 16)
        diag = torch.zeros((batch, DIAG_COUNT), dtype=torch.int64, device=cuda_dev)
        xh = f64(batch, nobs, n) if x_only else None
        need = _flps_ws(nobs, n, lag, batch, hess) or 256
        nb = need if ws_bytes is None else ws_bytes(need)
        ws = torch.empty(max(nb, 1), dtype=torch.uint8, device=cuda_dev)
        p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())   # noqa: E731
        rc = lib.pmmh_flps_model_batch_corr(model, p(obs), nobs, p(params), p(rvr), p(u), nobs, n, lag, batch, hess,
                                            p(filt), p(smo), p(ll), p(grad), p(traj), p(h1), p(h2), p(diag), p(xh),
                                            None, p(ws), nb, None)
        torch.cuda.synchronize()
        return rc

    big = (3 * (1 << 20)) // 2   # 1.5 M: a tile of N / SMs does not fit one CTA
    assert call(0, big, 30, 10, 1) == 1 and _flps_ws(30, big, 10, 1) is None and _filter_ws(30, big, 1) is None
    for lag in (1, 11):
        assert call(0, 1 << 14, 40, lag, 2) == 1 and _flps_ws(40, 1 << 14, lag, 2) is None
    assert call(0, 1 << 14, 19, 10, 2) == 1 and _flps_ws(19, 1 << 14, 10, 2) is None
    assert call(1, 1 << 14, 40, 10, 2, hess=1) == 1 and call(2, 1 << 14, 40, 10, 2, hess=1) == 1
    assert call(3, 1 << 14, 40, 10, 2) == 1 and call(-1, 1 << 14, 40, 10, 2) == 1
    assert call(0, 1 << 14, 40, 10, 2, x_only=True) == 1
    assert _flps_ws(40, 1 << 14, 10, 0) is None
    assert _filter_ws(1, 1 << 14, 2) is None and _filter_ws(40, 1 << 14, 0) is None
    # one byte short; the exact size runs
    assert call(0, 1 << 14, 40, 10, 2, ws_bytes=lambda need: need - 1) == 2
    assert call(0, 1 << 14, 40, 10, 2) == 0
    # the query: min(B, floor(SMs / G)) slices of the one-problem size with history
    for n, nobs, lag in ((1 << 14, 40, 10), (1 << 16, 30, 4), (4097, 50, 2)):
        G = min((n + 2047) // 2048, sm)
        one = ctypes.c_size_t()
        assert lib.pmmh_flps_model_workspace_bytes(nobs, n, lag, 1, ctypes.byref(one)) == 0
        fone = ctypes.c_size_t()
        assert lib.pmmh_filter_model_workspace_bytes(nobs, n, 1, ctypes.byref(fone)) == 0
        for batch in (1, 3, sm // G, sm // G + 5):
            slices = min(batch, sm // G)
            assert _flps_ws(nobs, n, lag, batch) == slices * one.value
            assert _filter_ws(nobs, n, batch) == slices * fone.value
            assert _flps_ws(nobs, n, lag, batch, 1) > _flps_ws(nobs, n, lag, batch)
