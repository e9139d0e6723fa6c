"""Batched backend of the lock-step sampler front-end (parameter/lockstep.py): the estimator calls of B
chains -- `smoother(model_k, rvs={'rvs': rvs_k})` with B different parameter vectors and B different u
(`mh_quasi_newton.py:331-335,376-380`) -- evaluated by ONE `pmmh_flps_sv_corr` launch over the batch
(chain kernel: one CTA per chain, N <= 4096; larger N runs the teams of the exchange / general kernels),
then published chain by chain with the host logic of `ParticleMethodsCUDA` (same `results` keys).

rvs per chain: a NumPy array in the reference's (NOBS, N+1) layout (stacked, uploaded, split on the device)
or a `DeviceRVS` handle.  Handles that are rows b = 0..B-1 of one [B, NOBS, N] tensor (as `BatchedRVSState`
hands them out) are used in place; others are stacked (one device copy).

pairing='exact' evaluates the batch with the SV model's exact fixed-lag smoother (model id 8, as
ParticleMethodsCUDA(pairing='exact')): one `pmmh_flps_model_corr` launch (chain kernel; the grid kernel for a
batch of one above 4096 particles), or one `pmmh_flps_model_batch_corr` launch (grid kernel, one team per chain)
when a chain wants the Hessian or a batch exceeds 4096 particles.
"""
import numpy as np
import torch
from scipy.stats import norm

from ... import kernels as K
from ..._lib import MODEL_SV_LEVERAGE_EXACT
from ...parameter.rvs import DeviceRVS
from .cuda import ParticleMethodsCUDA


class BatchedParticleMethodsCUDA(object):
    def __init__(self, model, no_particles=75, fixed_lag=10, device=None, verbose=False, pairing='reference'):
        self._one = ParticleMethodsCUDA(model, no_particles=no_particles, fixed_lag=fixed_lag, device=device,
                                        verbose=verbose, pairing=pairing)
        self.pairing = pairing
        self.template = self._one
        self.device = self._one.device
        self.alg_type = self._one.alg_type
        self.dim_rvs = self._one.dim_rvs
        self.settings = self._one.settings
        self.no_obs = self._one.no_obs
        self.no_particles = self._one.no_particles
        self._workspace = K.Workspace()
        self.no_launches = 0

    # ------------------------------------------------------------------ inputs
    def _stack_rvs(self, rvs_list):
        """-> (rvr [B, n_obs] device, u [B, n_obs, N] device)"""
        n_obs, n = self.no_obs, self.no_particles
        if all(isinstance(r, DeviceRVS) for r in rvs_list):
            us = [r.tensors['u'] for r in rvs_list]
            rr = [r.tensors['r_raw'] for r in rvs_list]
            base = us[0]._base if us[0]._base is not None else None
            step = n_obs * n * 8
            in_place = (base is not None and all(u._base is base for u in us) and
                        all(u.data_ptr() == us[0].data_ptr() + b * step for b, u in enumerate(us)) and
                        all(u.is_contiguous() for u in us))
            if in_place:
                u = torch.as_strided(us[0], (len(us), n_obs, n), (n_obs * n, n, 1))
            else:
                u = torch.stack(us)
            return K.norm_cdf(torch.stack(rr).contiguous()), u
        host = np.stack([np.ascontiguousarray(r, dtype=np.float64).reshape(-1) for r in rvs_list])
        if host.shape[1] != n_obs * (n + 1):
            raise ValueError("rvs has %d entries per chain, expected %d" % (host.shape[1], n_obs * (n + 1)))
        rv_r = norm.cdf(host[:, 0:n_obs])                      # bit-identical to cython.py:90 per chain
        d = torch.from_numpy(host).to(self.device)
        _, u = K.split_rvs(d, n_obs, n)
        return torch.from_numpy(np.ascontiguousarray(rv_r)).to(self.device), u

    def _evaluate_exact(self, obs_d, par, rvr, u, lag, hess):
        batch, n = u.shape[0], u.shape[2]
        if hess or (batch > 1 and n > 4096):
            out = K.flps_model_batch_corr(MODEL_SV_LEVERAGE_EXACT, obs_d, par, rvr, u, lag=lag, compute_hessian=hess,
                                          workspace=self._workspace)
        else:
            out = K.flps_model_corr(MODEL_SV_LEVERAGE_EXACT, obs_d, par, rvr, u, lag=lag, workspace=self._workspace)
        if not hess:
            out['hess1'] = out['hess2'] = torch.zeros((batch, 4, 4), dtype=torch.float64, device=self.device)
        return out

    # ------------------------------------------------------------------ the batch
    def evaluate_batch(self, requests):
        if not requests:
            return
        kinds = set(r.kind for r in requests)
        if kinds != {"smoother"}:
            raise NotImplementedError("the batched backend evaluates smoother calls (the quasi-Newton samplers' call)")
        try:
            models = [r.model for r in requests]
            hess = 1 if any(m.using_hessians for m in models) else 0
            _, obs_d = self._one._obs_device(models[0])
            params = np.stack([np.asarray(m.get_all_params(), dtype=np.float64) for m in models])
            rvs_list = []
            for r in requests:
                if 'rvs' in r.kwargs:
                    rvs_list.append(r.kwargs['rvs']['rvs'])
                else:
                    rvs_list.append(np.random.normal(size=self.dim_rvs))
            rvr, u = self._stack_rvs(rvs_list)
            par, lag = torch.from_numpy(params).to(self.device), self.settings['fixed_lag']
            if self.pairing == 'exact':
                out = self._evaluate_exact(obs_d, par, rvr, u, lag, hess)
            else:
                out = K.flps_sv_corr(obs_d, par, rvr, u, lag=lag, compute_hessian=hess, workspace=self._workspace)
            self.no_launches += 1
            host = {k: out[k].cpu().numpy() for k in ("filt", "smo", "log_like", "gradient", "traj", "hess1", "hess2", "diag")}
        except Exception as e:      # the whole batch failed: every chain rejects (cython.py:133-137 per chain)
            print("Error in CUDA code for the batched particle smoother.")
            print(e)
            for r in requests:
                r.ok, r.results = False, {}
            return
        for b, r in enumerate(requests):
            one = self._one
            one.results = {}
            one.settings.update(r.settings)
            try:
                r.ok = one._publish_smoother(r.model, host["filt"][b], host["smo"][b], host["log_like"][b:b + 1],
                                             host["gradient"][b], host["traj"][b], host["hess1"][b], host["hess2"][b],
                                             host["diag"][b])
            except Exception as e:
                print("Error in CUDA code for particle smoother.")
                print(e)
                r.ok = False
            r.results = dict(one.results)
            r.extra = dict(one.diagnostics)
