"""Particle methods on the GPU for the linear Gaussian state space model (``short_name == 'lgss'``):
x_t = phi x_{t-1} + sigma_v v_t, y_t = x_t + sigma_e e_t, x_0 = 0, parameters (phi, sigma_v, sigma_e); obs[0] is
not weighted.  The estimator contract is ``ParticleMethodsCUDA``'s (``filter`` / ``smoother`` -> bool, ``results``,
``settings``, ``dim_rvs``), so the samplers drive it unchanged.

``fully_adapted=True`` (default) runs the fully adapted particle filter with its fixed-lag gradient
(pmmh_flps_model_corr, model id 4): particles drawn from p(x_t | x_{t-1}, y_t) and weighted with p(y_{t+1} | x_t),
the likelihood estimate with the lowest variance of the filters here.  The kernel runs on the series shifted by one
(obs[1:]); the estimator adds log p(y_1) to ``log_like``, and the gradient already is that of the full
log-likelihood.  ``fully_adapted=False`` runs the bootstrap filter (model id 1) on the whole series.

``dim_rvs`` = (length of the series the kernel sees, N + 1): T - 1 rows when fully adapted, T otherwise.  ``rvs``
is that host array or a ``DeviceRVS`` of that shape, as for ``ParticleMethodsCUDA``.

``hessian=True`` (fully adapted only) lets the estimator serve second-order samplers: ``smoother`` with
``model.using_hessians`` runs model id 6 (pmmh_flps_model_batch_corr with compute_hessian, batch 1, on the grid
kernel) and publishes ``log_joint_hessian_estimate`` = hess1 + hess2 - g g' over (phi, sigma_v, sigma_e), g the summed
gradient slots (Louis' identity along the particles' genealogy; its variance grows with T / N).  Every other output is
model 4's.  Below 4097 particles a Hessian call runs on the grid kernel and a gradient-only call on the chain kernel,
so their log-likelihoods differ in the last bits.  With ``hessian=False`` (default) a call with ``model.using_hessians``
returns False.
"""
import numpy as np
import torch

from ... import kernels as K
from ..._lib import (DIAG_NEAR_TIES, DIAG_STATUS, MODEL_LINEAR_GAUSSIAN, MODEL_LINEAR_GAUSSIAN_FA_GRAD,
                     MODEL_LINEAR_GAUSSIAN_FA_HESS)
from ..base_state_inference import BaseStateInference
from .cuda import ParticleMethodsCUDA


def log_p_y1(y1, sigma_v, sigma_e):
    """log p(y_1) = log N(y_1; 0, sigma_v^2 + sigma_e^2) (x_0 = 0): the term the fully adapted filter's estimate
    of log p(y_2 .. y_T | y_1) lacks."""
    s2 = sigma_v * sigma_v + sigma_e * sigma_e
    return -0.5 * np.log(2.0 * np.pi * s2) - 0.5 * float(y1) ** 2 / s2


class LinearGaussianParticleMethodsCUDA(BaseStateInference):
    """Fully adapted (or bootstrap) particle filter and fixed-lag smoother of the linear Gaussian model (CUDA)."""

    # the same conversion of host arrays / DeviceRVS handles to the kernels' (rvr, u) as the SV estimator
    _rvs_device = ParticleMethodsCUDA._rvs_device
    _to_host = staticmethod(ParticleMethodsCUDA._to_host)

    def __init__(self, model, no_particles, fixed_lag=10, fully_adapted=True, device=None, hessian=False):
        if model.short_name != 'lgss':
            raise NameError("LinearGaussianParticleMethodsCUDA needs a linear Gaussian model ('lgss').")
        if hessian and not fully_adapted:
            raise ValueError("LinearGaussianParticleMethodsCUDA: the Hessian needs the fully adapted filter.")
        if not torch.cuda.is_available():
            raise RuntimeError("LinearGaussianParticleMethodsCUDA needs a CUDA device; there is no CPU fallback.")
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        self.fully_adapted = bool(fully_adapted)
        self.hessian = bool(hessian)
        self.model_id = MODEL_LINEAR_GAUSSIAN_FA_GRAD if self.fully_adapted else MODEL_LINEAR_GAUSSIAN
        self._workspace = K.Workspace()
        self._obs_cache = None
        no_particles, fixed_lag = int(no_particles), int(fixed_lag)
        series = model.no_obs + 1                       # T = len(obs)
        self.no_obs = series - 1 if self.fully_adapted else series   # what the kernel sees
        self.no_particles = no_particles
        self.dim_rvs = (self.no_obs, no_particles + 1)
        self.alg_type = 'particle'
        self.name = "Particle method (CUDA, %s) for %s model" % (
            "fully adapted" if self.fully_adapted else "bootstrap", model.short_name)
        self.settings = {'no_particles': no_particles,
                         'no_obs': self.no_obs,
                         'resampling_method': 'systematic',
                         'fixed_lag': fixed_lag,
                         'initial_state': 0.0,
                         'fully_adapted': self.fully_adapted,
                         'estimate_gradient': True,
                         'estimate_hessian': False}
        self.results = {}
        self.diagnostics = {}

    def _inputs(self, model, kwargs):
        """-> (obs on the device as the kernel sees it, params [1, 4] on the device, rvr, u, log p(y_1) or 0)"""
        obs = np.array(model.obs.flatten()).astype(float)
        if self._obs_cache is None or not np.array_equal(self._obs_cache[0], obs):
            seen = obs[1:] if self.fully_adapted else obs
            self._obs_cache = (obs, torch.from_numpy(np.ascontiguousarray(seen)).to(self.device))
        params = np.zeros(4)
        params[:3] = np.asarray(model.get_all_params(), dtype=np.float64)[:3]
        rvr, u = self._rvs_device(kwargs)
        extra = log_p_y1(obs[1], params[1], params[2]) if self.fully_adapted else 0.0
        return self._obs_cache[1], torch.from_numpy(params).reshape(1, 4).to(self.device), rvr, u, extra

    def _check_status(self, diag):
        self.diagnostics = {'near_ties': int(diag[DIAG_NEAR_TIES]), 'status': int(diag[DIAG_STATUS])}
        if int(diag[DIAG_STATUS]) != 0:
            raise FloatingPointError("degenerate particle cloud")

    def filter(self, model, **kwargs):
        """The particle filter alone (pmmh_filter_model_corr): log_like, filt_state_est, state_trajectory."""
        try:
            obs_d, par_d, rvr, u, extra = self._inputs(model, kwargs)
            out = K.filter_model_corr(self.model_id, obs_d, par_d, rvr, u, workspace=self._workspace)
            xf, ll, xtraj, diag = self._to_host([out['filt'][0], out['log_like'], out['traj'][0], out['diag'][0]])
            self._check_status(diag)
            self.results.update({'filt_state_est': np.array(xf).flatten()})
            self.results.update({'state_trajectory': np.array(xtraj).flatten()})
            self.results.update({'log_like': float(ll[0]) + extra})
            return True
        except Exception as e:
            print("Error in CUDA code for particle filter.")
            print(e)
            return False

    def smoother(self, model, **kwargs):
        """Fixed-lag smoother (pmmh_flps_model_corr): log_like, filtered / smoothed states, trajectory and the
        gradient estimate (the sum of gradient rows 0..2 over the slots, non-finite entries taken as 0).  With
        ``model.using_hessians`` (``hessian=True`` only) pmmh_flps_model_batch_corr with the Hessian branch, and the
        Hessian estimate hess1 + hess2 - g g'."""
        if model.using_hessians and not self.hessian:
            print("LinearGaussianParticleMethodsCUDA: no Hessian estimate (construct it with hessian=True).")
            return False
        try:
            obs_d, par_d, rvr, u, extra = self._inputs(model, kwargs)
            hess = bool(model.using_hessians)
            self.settings['estimate_hessian'] = hess
            if hess:
                out = K.flps_model_batch_corr(MODEL_LINEAR_GAUSSIAN_FA_HESS, obs_d, par_d, rvr, u,
                                              lag=self.settings['fixed_lag'], compute_hessian=1,
                                              workspace=self._workspace)
            else:
                out = K.flps_model_corr(self.model_id, obs_d, par_d, rvr, u, lag=self.settings['fixed_lag'],
                                        workspace=self._workspace)
            tensors = [out['filt'][0], out['smo'][0], out['log_like'], out['gradient'][0], out['traj'][0], out['diag'][0]]
            if hess:
                tensors += [out['hess1'][0], out['hess2'][0]]
            xf, xs, ll, grad, xtraj, diag, *h12 = self._to_host(tensors)
            self._check_status(diag)
            self.results.update({'filt_state_est': np.array(xf).flatten()})
            self.results.update({'state_trajectory': np.array(xtraj).flatten()})
            self.results.update({'smo_state_est': np.array(xs).flatten()})
            self.results.update({'log_like': float(ll[0]) + extra})
            if model.using_gradients or hess:
                g = np.array(grad[:3], dtype=np.float64)
                g[~np.isfinite(g)] = 0.0
                self.results.update({'log_joint_gradient_estimate': g.sum(axis=1)})
            if hess:
                g = self.results['log_joint_gradient_estimate']
                self.results.update({'log_joint_hessian_estimate': (h12[0] + h12[1])[:3, :3] - np.outer(g, g)})
            return self._estimate_gradient_and_hessian(model)
        except Exception as e:
            print("Error in CUDA code for particle smoother.")
            print(e)
            return False
