"""Thin torch-facing wrappers over the C ABI (include/pmmh_qn.h).

Tensors are float64 / int32 / int64 CUDA tensors; PyTorch only allocates them and owns the
stream the kernels are enqueued on (``torch.cuda.current_stream()``).  Everything here is
asynchronous; nothing falls back to the CPU.
"""
import ctypes

import torch

from . import _lib

_F64 = torch.float64


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.PmmhError("expected CUDA tensors (there is no CPU path)")
        if not t.is_contiguous():
            raise _lib.PmmhError("expected contiguous tensors")


class Workspace(object):
    """A reusable, growing device scratch buffer (one per estimator)."""

    def __init__(self):
        self.buf = None

    def get(self, nbytes, device):
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != device:
            self.buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        return self.buf


def device_info():
    lib = _lib.load()
    sm, major, minor = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _lib.check(lib.pmmh_device_info(ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor)),
               "pmmh_device_info")
    return sm.value, major.value, minor.value


def set_sv_algorithm(algorithm):
    """0 = automatic (chain / grid / streaming / exchange kernel where eligible, the general kernel
    otherwise and as their fallback), 1 = general kernel only, 2 / 3 = exchange / chain kernel without
    the general-kernel fallback, 4 / 5 = streaming kernels with records / with path storage, 6 = grid
    kernel (pmmh_sv_set_algorithm; the selection table is in include/pmmh_qn.h)."""
    lib = _lib.load()
    _lib.check(lib.pmmh_sv_set_algorithm(int(algorithm)), "pmmh_sv_set_algorithm")


def sv_workspace_bytes(n_obs, n_particles, lag, batch, compute_hessian, mode=0, have_history=False,
                       ctas_per_problem=0):
    lib = _lib.load()
    out = ctypes.c_size_t()
    _lib.check(lib.pmmh_sv_workspace_bytes(n_obs, n_particles, lag, batch, int(bool(compute_hessian)),
                                           mode, int(bool(have_history)), ctas_per_problem,
                                           ctypes.byref(out)), "pmmh_sv_workspace_bytes")
    return out.value


def _sv_common(obs, params, rvr, u):
    _need_cuda(obs, params, rvr, u)
    if u.dim() == 2:
        u = u.unsqueeze(0)
    batch, n_obs, n = u.shape
    params = params.reshape(batch, 4)
    rvr = rvr.reshape(batch, n_obs)
    if obs.dim() == 1:
        obs_stride = 0
        assert obs.shape[0] == n_obs
    else:
        assert obs.shape == (batch, n_obs)
        obs_stride = n_obs
    for t in (obs, params, rvr, u):
        assert t.dtype == _F64
    return obs, obs_stride, params, rvr, u, batch, n_obs, n


def _sv_outputs(dev, batch, n_obs, n=0, smoother=True, hessian=False, history=False):
    """Output tensors of the smoother / filter entries: filt, (smo), log_like, (gradient), traj, (hess1, hess2),
    diag and, with history, X / A [B, n_obs, N]."""
    def f64(*shape):
        return torch.empty(shape, dtype=_F64, device=dev)
    out = {"filt": f64(batch, n_obs)}
    if smoother:
        out["smo"] = f64(batch, n_obs)
    out["log_like"] = f64(batch)
    if smoother:
        out["gradient"] = f64(batch, 4, n_obs)
    out["traj"] = f64(batch, n_obs)
    if hessian:
        out["hess1"] = f64(batch, 4, 4)
        out["hess2"] = f64(batch, 4, 4)
    out["diag"] = torch.zeros((batch, _lib.DIAG_COUNT), dtype=torch.int64, device=dev)
    if history:
        out["X"] = f64(batch, n_obs, n)
        out["A"] = torch.empty((batch, n_obs, n), dtype=torch.int32, device=dev)
    return out


def flps_sv_corr(obs, params, rvr, u, lag=10, compute_hessian=False, store_history=False,
                 ctas_per_problem=0, workspace=None):
    """Fixed-lag particle smoother (pmmh_flps_sv_corr).  u is time-major [B, n_obs, N].
    Returns a dict of device tensors."""
    lib = _lib.load()
    obs, obs_stride, params, rvr, u, batch, n_obs, n = _sv_common(obs, params, rvr, u)
    dev = u.device
    hess = int(bool(compute_hessian))
    out = _sv_outputs(dev, batch, n_obs, n, hessian=True, history=store_history)
    xh, ah = out.get("X"), out.get("A")
    nbytes = sv_workspace_bytes(n_obs, n, lag, batch, hess, 0, store_history, ctas_per_problem)
    ws = (workspace or Workspace()).get(nbytes, dev)
    _lib.check(lib.pmmh_flps_sv_corr(
        _ptr(obs), obs_stride, _ptr(params), _ptr(rvr), _ptr(u), n_obs, n, lag, batch, hess,
        _ptr(out["filt"]), _ptr(out["smo"]), _ptr(out["log_like"]), _ptr(out["gradient"]),
        _ptr(out["traj"]), _ptr(out["hess1"]), _ptr(out["hess2"]), _ptr(out["diag"]),
        _ptr(xh), _ptr(ah), _ptr(ws), ws.numel(), ctas_per_problem, _stream()), "pmmh_flps_sv_corr")
    out["_workspace"] = ws
    return out


def _workspace_bytes(query, *sizes):
    wb = ctypes.c_size_t()
    _lib.check(getattr(_lib.load(), query)(*sizes, ctypes.byref(wb)), query)
    return wb.value


def _model_corr(name, model_id, obs, params, rvr, u, lag, hess, store_history, workspace):
    """pmmh_<name>_corr after its workspace query pmmh_<name>_workspace_bytes: the smoother (name flps_model or
    flps_model_batch) or the filter alone (filter_model or filter_model_batch)"""
    lib = _lib.load()
    obs, obs_stride, params, rvr, u, batch, n_obs, n = _sv_common(obs, params, rvr, u)
    dev = u.device
    smoother, batched = name.startswith("flps"), name.endswith("batch")
    out = _sv_outputs(dev, batch, n_obs, n, smoother=smoother, hessian=bool(hess), history=store_history)
    sizes = [n_obs, n] + ([lag] if smoother else []) + [batch] + ([hess] if smoother and batched else [])
    ws = (workspace or Workspace()).get(_workspace_bytes("pmmh_%s_workspace_bytes" % name, *sizes), dev)
    keys = ["filt", "smo", "log_like", "gradient", "traj"] if smoother else ["filt", "log_like", "traj"]
    if smoother and batched:
        keys += ["hess1", "hess2"]
    outs = [_ptr(out.get(k)) for k in keys + ["diag", "X", "A"]]
    entry = "pmmh_%s_corr" % name
    _lib.check(getattr(lib, entry)(int(model_id), _ptr(obs), obs_stride, _ptr(params), _ptr(rvr), _ptr(u), *sizes,
                                   *outs, _ptr(ws), ws.numel(), _stream()), entry)
    out["_workspace"] = ws
    return out


def flps_model_corr(model_id, obs, params, rvr, u, lag=10, store_history=False, workspace=None):
    """Model-generic fixed-lag smoother (pmmh_flps_model_corr, csrc/pf_model.cuh): log-likelihood +
    gradient of [B] problems.  2 <= lag <= 10.  Up to 4096 particles: any B, one CTA per problem (chain
    kernel, diag kernel 3).  Above: B == 1, n_obs >= 2 lag and up to 7168 particles per SM (1,060,864 on
    148 SMs), one persistent launch over the GPU (grid kernel, diag kernel 5).  Other sizes raise PmmhError.
    ``model_id``: _lib.MODEL_SV_LEVERAGE (bit-identical to flps_sv_corr on the same kernel),
    _lib.MODEL_LINEAR_GAUSSIAN, _lib.MODEL_LINEAR_GAUSSIAN_FA, _lib.MODEL_LINEAR_GAUSSIAN_FA_GRAD or
    _lib.MODEL_LINEAR_GAUSSIAN_FA_HESS; params [B, 4] (unused slots ignored).  The fully adapted models 2, 4 and 6 take
    the series shifted by one (obs[1:]) and their log_like lacks log p(y_1); model 4 adds model 2 a gradient whose slot
    k holds the contribution of obs[1:][k], so that the slots sum to the score of the full log-likelihood
    (include/pmmh_qn.h).  Model 6 is model 4 here, bit for bit (its Hessian: flps_model_batch_corr).
    _lib.MODEL_SV_LEVERAGE_EXACT (8) runs model 0's particle system on the same inputs (filt, log_like, traj, diag and
    history bit-identical) with the exact fixed-lag score: slot k holds the transition (x_k, x_k+1) scored with obs[k],
    the slots sum to an estimate of the score of log_like (its Hessian: flps_model_batch_corr).
    No fallback pass: diag[:, PMMH_DIAG_STATUS] == 1 reports an abandoned evaluation."""
    return _model_corr("flps_model", model_id, obs, params, rvr, u, lag, 0, store_history, workspace)


def filter_model_corr(model_id, obs, params, rvr, u, store_history=False, workspace=None):
    """Model-generic particle filter (pmmh_filter_model_corr): log-likelihood, filtered means, trajectory and
    diag of [B] problems without the fixed-lag smoother -- bit-identical to those outputs of flps_model_corr
    for any lag.  Up to 4096 particles: any B (chain kernel, diag kernel 3).  Above: B == 1 and up to 7168
    particles per SM (grid kernel, diag kernel 5).  n_obs >= 2; other sizes raise PmmhError.  ``model_id`` and
    params as for flps_model_corr (models 4 and 6 run model 2's filter, model 8 model 0's).  No fallback pass: diag[:, PMMH_DIAG_STATUS] == 1 reports an abandoned
    evaluation."""
    return _model_corr("filter_model", model_id, obs, params, rvr, u, 2, 0, store_history, workspace)


def flps_model_batch_workspace_bytes(n_obs, n_particles, lag, batch, compute_hessian=0):
    return _workspace_bytes("pmmh_flps_model_batch_workspace_bytes", n_obs, n_particles, lag, batch,
                            int(bool(compute_hessian)))


def filter_model_batch_workspace_bytes(n_obs, n_particles, batch):
    return _workspace_bytes("pmmh_filter_model_batch_workspace_bytes", n_obs, n_particles, batch)


def flps_model_batch_corr(model_id, obs, params, rvr, u, lag=10, compute_hessian=0, store_history=False,
                          workspace=None):
    """Batch of [B] problems on the grid kernel, one team of CTAs per problem (pmmh_flps_model_batch_corr): the
    outputs of problem b are bit-identical to flps_model_corr on that problem alone with B == 1 (and, for
    _lib.MODEL_SV_LEVERAGE, to flps_sv_corr on the grid kernel, also with the Hessian).  Any B on every shape the
    one-problem grid run takes (above 4096 particles: n_obs >= 2 lag, up to 7168 particles per CTA of
    ceil(N / 2048)); model ids as for flps_model_corr; compute_hessian for _lib.MODEL_SV_LEVERAGE (the reference's
    Hessian branch) and _lib.MODEL_LINEAR_GAUSSIAN_FA_HESS (Louis' identity on model 4's pairs and weights:
    hess1 + hess2 - g g', g = the summed gradient slots, estimates the Hessian of the full log-likelihood over
    (phi, sigma_v, sigma_e); row and column 3 are 0), and _lib.MODEL_SV_LEVERAGE_EXACT (the same identity on model 8's
    pairs, over (mu, atanh phi, log sigma_v, atanh rho)).  Every other output of model 6 is model 4's, bit for bit, with
    compute_hessian 0 or 1.  Returns the dict of flps_model_corr, plus hess1 / hess2 [B, 4, 4] with compute_hessian.  No fallback pass: diag[:, PMMH_DIAG_STATUS] == 1 reports an abandoned
    problem, the others are unaffected."""
    return _model_corr("flps_model_batch", model_id, obs, params, rvr, u, lag, int(bool(compute_hessian)),
                       store_history, workspace)


def filter_model_batch_corr(model_id, obs, params, rvr, u, store_history=False, workspace=None):
    """Batch of [B] particle filters on the grid kernel, one team of CTAs per problem
    (pmmh_filter_model_batch_corr): the outputs of problem b are bit-identical to filter_model_corr on that problem
    alone (and to those outputs of flps_model_batch_corr).  Any B where a tile of the one-problem grid run fits one
    CTA, n_obs >= 2.  Returns the dict of filter_model_corr."""
    return _model_corr("filter_model_batch", model_id, obs, params, rvr, u, 2, 0, store_history, workspace)


def flps_sv_corr_philox(obs, params, rvr, seed, philox_offset, n_particles, lag=10, workspace=None):
    """Log-likelihood + gradient of one problem whose auxiliary variables are a Philox stream
    (pmmh_flps_sv_corr_philox): any N on one device without ever storing u."""
    lib = _lib.load()
    _need_cuda(obs, params, rvr)
    dev = obs.device
    n_obs = obs.shape[0]
    out = _sv_outputs(dev, 1, n_obs)
    nb = ctypes.c_size_t()
    _lib.check(lib.pmmh_flps_sv_corr_philox_workspace_bytes(n_obs, int(n_particles), int(lag), ctypes.byref(nb)),
               "pmmh_flps_sv_corr_philox_workspace_bytes")
    ws = (workspace or Workspace()).get(nb.value, dev)
    _lib.check(lib.pmmh_flps_sv_corr_philox(
        _ptr(obs), _ptr(params.reshape(-1)), _ptr(rvr.reshape(-1)), int(seed), int(philox_offset), n_obs,
        int(n_particles), int(lag), _ptr(out["filt"]), _ptr(out["smo"]), _ptr(out["log_like"]),
        _ptr(out["gradient"]), _ptr(out["traj"]), _ptr(out["diag"]), _ptr(ws), ws.numel(), _stream()),
        "pmmh_flps_sv_corr_philox")
    out["_workspace"] = ws
    return out


def sv_streamed_eligible(n_obs, n_particles, lag=10, ctas_per_problem=0):
    """True if pmmh_flps_sv_corr_streamed takes these sizes under the current algorithm (a grid,
    exchange or streaming kernel is selected for them)."""
    return bool(_lib.load().pmmh_sv_streamed_eligible(int(n_obs), int(n_particles), int(lag),
                                                      int(ctas_per_problem)))


def flps_sv_corr_streamed(rvs_host, obs, params, rvr, n_obs, n_particles, lag=10, ctas_per_problem=0,
                          workspace=None, stage=None):
    """Log-likelihood + gradient with the auxiliary variables still in host memory
    (pmmh_flps_sv_corr_streamed): ``rvs_host`` is the reference's (n_obs, N+1) float64 array
    (C-contiguous NumPy array; pinned memory makes the copies overlap the kernel).  The caller
    must keep ``rvs_host`` alive and unchanged until the stream has been synchronised."""
    lib = _lib.load()
    _need_cuda(obs, params, rvr)
    if rvs_host.dtype != "float64" or not rvs_host.flags["C_CONTIGUOUS"] or rvs_host.size != n_obs * (n_particles + 1):
        raise _lib.PmmhError("flps_sv_corr_streamed: rvs must be a C-contiguous float64 (n_obs, N+1) array")
    dev = obs.device
    params = params.reshape(1, 4)
    rvr = rvr.reshape(1, n_obs)
    out = _sv_outputs(dev, 1, n_obs, hessian=True)
    wb = ctypes.c_size_t()
    _lib.check(lib.pmmh_sv_streamed_workspace_bytes(n_obs, n_particles, lag, ctas_per_problem, ctypes.byref(wb)),
               "pmmh_sv_streamed_workspace_bytes")
    ws = (workspace or Workspace()).get(wb.value, dev)
    sb = ctypes.c_size_t()
    _lib.check(lib.pmmh_sv_stage_bytes(n_obs, n_particles, ctypes.byref(sb)), "pmmh_sv_stage_bytes")
    st = (stage or Workspace()).get(sb.value, dev)
    _lib.check(lib.pmmh_flps_sv_corr_streamed(
        ctypes.c_void_p(rvs_host.ctypes.data), _ptr(obs), _ptr(params), _ptr(rvr), n_obs, n_particles, lag,
        _ptr(st), st.numel(), _ptr(out["filt"]), _ptr(out["smo"]), _ptr(out["log_like"]),
        _ptr(out["gradient"]), _ptr(out["traj"]), _ptr(out["hess1"]), _ptr(out["hess2"]),
        _ptr(out["diag"]), _ptr(ws), ws.numel(), ctas_per_problem, _stream()), "pmmh_flps_sv_corr_streamed")
    out["_workspace"] = ws
    out["_stage"] = st
    return out


def bpf_sv_corr(obs, params, rvr, u, read_mode=_lib.BPF_PARITY, store_history=False,
                ctas_per_problem=0, workspace=None):
    """Bootstrap particle filter (pmmh_bpf_sv_corr)."""
    lib = _lib.load()
    obs, obs_stride, params, rvr, u, batch, n_obs, n = _sv_common(obs, params, rvr, u)
    dev = u.device
    out = _sv_outputs(dev, batch, n_obs, n, smoother=False, history=store_history)
    xh, ah = out.get("X"), out.get("A")
    nbytes = sv_workspace_bytes(n_obs, n, 2, batch, 0, 1, store_history, ctas_per_problem)
    ws = (workspace or Workspace()).get(nbytes, dev)
    _lib.check(lib.pmmh_bpf_sv_corr(
        _ptr(obs), obs_stride, _ptr(params), _ptr(rvr), _ptr(u), n_obs, n, batch, read_mode,
        _ptr(out["filt"]), _ptr(out["log_like"]), _ptr(out["traj"]), _ptr(out["diag"]),
        _ptr(xh), _ptr(ah), _ptr(ws), ws.numel(), ctas_per_problem, _stream()), "pmmh_bpf_sv_corr")
    out["_workspace"] = ws
    return out


def split_rvs(rvs, n_obs, n_particles):
    """rvs [B, n_obs, N+1] (or [n_obs, N+1]) -> (r_raw [B, n_obs], u [B, n_obs, N] time-major)."""
    lib = _lib.load()
    _need_cuda(rvs)
    per = n_obs * (n_particles + 1)
    batch = rvs.numel() // per
    if batch * per != rvs.numel() or batch < 1 or rvs.dtype != _F64:
        raise _lib.PmmhError("split_rvs: expected float64 rvs with a multiple of n_obs*(N+1) entries")
    r_raw = torch.empty((batch, n_obs), dtype=_F64, device=rvs.device)
    u = torch.empty((batch, n_obs, n_particles), dtype=_F64, device=rvs.device)
    _lib.check(lib.pmmh_split_rvs(_ptr(rvs), n_obs, n_particles, batch, _ptr(r_raw), _ptr(u),
                                  _stream()), "pmmh_split_rvs")
    return r_raw, u


def norm_cdf(x, out=None):
    lib = _lib.load()
    _need_cuda(x)
    if out is None:
        out = torch.empty_like(x)
    _lib.check(lib.pmmh_norm_cdf(_ptr(x), _ptr(out), x.numel(), _stream()), "pmmh_norm_cdf")
    return out


def importance_discrete(obs, params, rvr, rvp, n_obs, n_particles):
    """Random-effects importance sampler; rvp [B, n_obs*N] in the reference's flat layout."""
    lib = _lib.load()
    _need_cuda(obs, params, rvr, rvp)
    batch = rvp.numel() // (n_obs * n_particles)
    assert rvp.numel() == batch * n_obs * n_particles
    dev = rvp.device
    obs_stride = 0 if obs.dim() == 1 else n_obs
    out = {
        "filt": torch.empty((batch, n_obs), dtype=_F64, device=dev),
        "log_like": torch.empty((batch,), dtype=_F64, device=dev),
        "traj": torch.empty((batch, n_obs), dtype=_F64, device=dev),
        "gradient": torch.empty((batch, 2), dtype=_F64, device=dev),
        "traj_idx": torch.empty((batch,), dtype=torch.int32, device=dev),
    }
    _lib.check(lib.pmmh_importance_discrete(
        _ptr(obs), obs_stride, _ptr(params), _ptr(rvr), _ptr(rvp), n_obs, n_particles, batch,
        _ptr(out["filt"]), _ptr(out["log_like"]), _ptr(out["traj"]), _ptr(out["gradient"]),
        _ptr(out["traj_idx"]), _stream()), "pmmh_importance_discrete")
    return out


def crank_nicolson(u, sigma_u, xi=None, seed=0, philox_offset=0, out=None):
    """u' = sqrt(1 - sigma_u^2) u + sigma_u xi; xi=None draws Philox normals on the device."""
    lib = _lib.load()
    _need_cuda(u, xi)
    if out is None:
        out = torch.empty_like(u)
    _lib.check(lib.pmmh_crank_nicolson(_ptr(u), _ptr(xi), _ptr(out), u.numel(), float(sigma_u),
                                       int(seed), int(philox_offset), _stream()), "pmmh_crank_nicolson")
    return out


def subsample_indices(u, n_data, apply_cdf=True, want_sorted=False, workspace=None):
    """sort(Phi(u)) + stratified indices (state/direct/standard.py:75-76)."""
    lib = _lib.load()
    _need_cuda(u)
    m = u.numel()
    dev = u.device
    nb = ctypes.c_size_t()
    _lib.check(lib.pmmh_subsample_workspace_bytes(m, ctypes.byref(nb)), "pmmh_subsample_workspace_bytes")
    ws = (workspace or Workspace()).get(nb.value, dev)
    idx = torch.empty((m,), dtype=torch.int32, device=dev)
    srt = torch.empty((m,), dtype=_F64, device=dev) if want_sorted else None
    _lib.check(lib.pmmh_subsample_indices(_ptr(u), m, int(n_data), int(bool(apply_cdf)), _ptr(idx),
                                          _ptr(srt), _ptr(ws), ws.numel(), _stream()),
               "pmmh_subsample_indices")
    return (idx, srt) if want_sorted else idx


def logistic_loglike(x, y, idx, beta, compute_hessian=False, row_begin=0, row_end=None,
                     workspace=None):
    """Subsampled logistic log-lik / gradient / Hessian.  Returns a device vector
    [1 + d + d*d]: log_like, gradient, hessian (row-major)."""
    lib = _lib.load()
    _need_cuda(x, y, idx, beta)
    d = x.shape[1]
    m = idx.numel()
    if row_end is None:
        row_end = row_begin + x.shape[0]
    hess = int(bool(compute_hessian))
    nb = ctypes.c_size_t()
    _lib.check(lib.pmmh_logistic_workspace_bytes(m, d, hess, ctypes.byref(nb)),
               "pmmh_logistic_workspace_bytes")
    ws = (workspace or Workspace()).get(nb.value, x.device)
    out = torch.empty((1 + d + d * d,), dtype=_F64, device=x.device)
    _lib.check(lib.pmmh_logistic_loglike(_ptr(x), _ptr(y), _ptr(idx), m, d, int(row_begin),
                                         int(row_end), _ptr(beta), hess, _ptr(out), _ptr(ws),
                                         ws.numel(), _stream()), "pmmh_logistic_loglike")
    return out
