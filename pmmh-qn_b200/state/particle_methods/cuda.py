"""Particle methods on the GPU -- drop-in for the reference's ``ParticleMethodsCython``
(/root/reference/python/state/particle_methods/cython.py:30-168).

Same contract: ``filter(model, **kw) -> bool``, ``smoother(model, **kw) -> bool``, results in
``self.results`` under the reference's keys, ``settings`` / ``dim_rvs`` / ``alg_type`` as the
samplers read them (parameter/mcmc/base_class.py:100-101,169-183).  The reference bakes
NPART / NOBS / LAG into its Cython module at compile time
(stochastic_volatility.pyx:17-19); here they are constructor arguments.

``pairing='exact'`` runs the SV model's exact fixed-lag smoother instead (model id 8,
include/pmmh_qn.h PMMH_MODEL_SV_LEVERAGE_EXACT): the same particle system, with every transition
scored against its own leverage observation, and a Hessian by Louis' identity published as
hess1 + hess2 - g g'.  The default ``'reference'`` reproduces the reference, quirks Q5 / Q6 / Q9
included.

``rvs={'rvs': x}`` accepts either the reference's (n_obs, N+1) NumPy array or a device-resident
``DeviceRVS`` handle (pmmh-qn_b200/parameter/rvs.py).  Without ``rvs`` fresh normals are drawn
as the reference does (cython.py:60,93).
"""
import numpy as np
import torch
from scipy.stats import norm

from ... import kernels as K
from ..._lib import BPF_INTENDED, BPF_PARITY, DIAG_NEAR_TIES, DIAG_STATUS, MODEL_SV_LEVERAGE_EXACT, PmmhError
from ...parameter.rvs import DeviceRVS
from ..base_state_inference import BaseStateInference


class ParticleMethodsCUDA(BaseStateInference):
    """Bootstrap particle filter and fixed-lag particle smoother (CUDA, sm_100a)."""

    def __init__(self, model, no_particles=75, fixed_lag=10, device=None,
                 bpf_read_mode='parity', ctas_per_problem=0, verbose=False, pairing='reference'):
        self.alg_type = 'particle'
        if model.short_name != 'sv':
            raise NameError("CUDA implementation for model missing.")
        if pairing not in ('reference', 'exact'):
            raise ValueError("pairing must be 'reference' or 'exact'")
        if not torch.cuda.is_available():
            raise RuntimeError("ParticleMethodsCUDA needs a CUDA device; there is no CPU fallback.")
        self.pairing = pairing
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        self.bpf_read_mode = {'parity': BPF_PARITY, 'intended': BPF_INTENDED}[bpf_read_mode]
        self.ctas_per_problem = int(ctas_per_problem)
        self._workspace = K.Workspace()
        self._stage = K.Workspace()
        self.stream_min_particles = 1 << 15   # below this the upload is too small to be worth overlapping
        self._obs_cache = None
        self._init_particle_method(model, int(no_particles), int(fixed_lag), verbose)
        if pairing == 'exact':
            self._check_exact_sizes(model)
        self.results = {}
        self.diagnostics = {}

    # ------------------------------------------------------------------ helpers
    def _obs_device(self, model):
        # (the comparison reads n_obs doubles per call: the observations may be replaced on the model
        # between calls, and n_obs is ~1e3)
        obs = np.array(model.obs.flatten()).astype(float)
        if self._obs_cache is None or not np.array_equal(self._obs_cache[0], obs):
            self._obs_cache = (obs, torch.from_numpy(obs).to(self.device))
        return obs, self._obs_cache[1]

    def _rvs_device(self, kwargs):
        """-> (rvr [n_obs] device, u [n_obs, N] device time-major)"""
        n_obs, n = self.no_obs, self.no_particles
        rvs = kwargs['rvs']['rvs'] if 'rvs' in kwargs else np.random.normal(size=self.dim_rvs)
        if isinstance(rvs, DeviceRVS):
            rvr = K.norm_cdf(rvs.tensors['r_raw'])
            u = rvs.tensors['u']
            return rvr, u
        rvs = np.ascontiguousarray(rvs, dtype=np.float64)
        if rvs.size != n_obs * (n + 1):
            raise ValueError("rvs has %d entries, expected %d" % (rvs.size, n_obs * (n + 1)))
        flat = rvs.reshape(-1)
        # Phi of the first n_obs FLAT entries on the host: bit-identical to cython.py:90
        rv_r = norm.cdf(flat[0:n_obs]).flatten()
        d = torch.from_numpy(flat).to(self.device, non_blocking=True)
        _, u = K.split_rvs(d, n_obs, n)
        rvr = torch.from_numpy(rv_r).to(self.device, non_blocking=True)
        return rvr, u[0]

    def _smoother_streamed(self, rvs, obs_d, params):
        """Large host-resident rvs: let the copy engine feed the running kernel
        (pmmh_flps_sv_corr_streamed) instead of upload -> layout kernel -> smoother.  Returns
        None when this path does not apply or the kernel abandoned the evaluation."""
        n_obs, n = self.no_obs, self.no_particles
        lag = self.settings['fixed_lag']
        if not isinstance(rvs, np.ndarray) or n < self.stream_min_particles:
            return None
        if rvs.dtype != np.float64 or not rvs.flags['C_CONTIGUOUS'] or rvs.size != n_obs * (n + 1):
            return None
        if not K.sv_streamed_eligible(n_obs, n, lag, self.ctas_per_problem):
            return None
        flat = rvs.reshape(-1)
        rv_r = norm.cdf(flat[0:n_obs]).flatten()   # bit-identical to cython.py:90
        rvr = torch.from_numpy(rv_r).to(self.device, non_blocking=True)
        try:
            out = K.flps_sv_corr_streamed(rvs, obs_d, torch.from_numpy(params).to(self.device), rvr, n_obs, n,
                                          lag=lag, ctas_per_problem=self.ctas_per_problem,
                                          workspace=self._workspace, stage=self._stage)
        except PmmhError:      # a size / workspace the streamed entry point refuses: upload instead
            return None
        if int(out['diag'][0, DIAG_STATUS].item()) != 0:   # synchronises; abandoned: use the general path
            return None
        return out

    def _check_exact_sizes(self, model):
        """raises PmmhError on the sizes the model entries refuse (the smoother's; the Hessian's when the model asks
        for it)"""
        n_obs, n, lag = self.no_obs, self.no_particles, self.settings['fixed_lag']
        if n_obs < lag + 1:
            raise PmmhError("pairing='exact' needs n_obs >= lag + 1")
        K._workspace_bytes("pmmh_flps_model_workspace_bytes", n_obs, n, lag, 1)
        if model.using_hessians:
            K._workspace_bytes("pmmh_flps_model_batch_workspace_bytes", n_obs, n, lag, 1, 1)

    def _smoother_exact(self, obs_d, params, hessian_flag, kwargs):
        """model 8 on the uploaded rvs: flps_model_corr, or flps_model_batch_corr with the Hessian"""
        rvr, u = self._rvs_device(kwargs)
        par = torch.from_numpy(params).to(self.device)
        lag = self.settings['fixed_lag']
        if hessian_flag:
            return K.flps_model_batch_corr(MODEL_SV_LEVERAGE_EXACT, obs_d, par, rvr, u, lag=lag, compute_hessian=1,
                                           workspace=self._workspace)
        out = K.flps_model_corr(MODEL_SV_LEVERAGE_EXACT, obs_d, par, rvr, u, lag=lag, workspace=self._workspace)
        out['hess1'] = out['hess2'] = torch.zeros((1, 4, 4), dtype=torch.float64, device=self.device)
        return out

    @staticmethod
    def _to_host(tensors):
        flat = torch.cat([t.reshape(-1).to(torch.float64) for t in tensors]).cpu().numpy()
        out, off = [], 0
        for t in tensors:
            out.append(flat[off:off + t.numel()].reshape(tuple(t.shape)))
            off += t.numel()
        return out

    # ------------------------------------------------------------------ filter
    def filter(self, model, **kwargs):
        """Bootstrap particle filter (bpf_sv_corr, stochastic_volatility.pyx:61-201)."""
        try:
            _, obs_d = self._obs_device(model)
            params = np.asarray(model.get_all_params(), dtype=np.float64)
            rvr, u = self._rvs_device(kwargs)
            out = K.bpf_sv_corr(obs_d, torch.from_numpy(params).to(self.device), rvr, u,
                                read_mode=self.bpf_read_mode, ctas_per_problem=self.ctas_per_problem,
                                workspace=self._workspace)
            xf, ll, xtraj, diag = self._to_host([out['filt'][0], out['log_like'], out['traj'][0],
                                                 out['diag'][0]])
            self.diagnostics = {'near_ties': int(diag[DIAG_NEAR_TIES]), 'status': int(diag[DIAG_STATUS])}
            if int(diag[DIAG_STATUS]) != 0:
                raise FloatingPointError("degenerate particle cloud")
            self.results.update({'filt_state_est': np.array(xf).flatten()})
            self.results.update({'state_trajectory': np.array(xtraj).flatten()})
            self.results.update({'log_like': float(ll[0])})
            return True
        except Exception as e:
            print("Error in CUDA code for particle filter.")
            print(e)
            return False

    # ---------------------------------------------------------------- smoother
    def smoother(self, model, **kwargs):
        """Fixed-lag particle smoother (flps_sv_corr, stochastic_volatility.pyx:205-655)."""
        hessian_flag = 1 if model.using_hessians else 0
        try:
            _, obs_d = self._obs_device(model)
            params = np.asarray(model.get_all_params(), dtype=np.float64)
            out = None
            if self.pairing == 'exact':
                out = self._smoother_exact(obs_d, params, hessian_flag, kwargs)
            elif not hessian_flag and 'rvs' in kwargs:
                out = self._smoother_streamed(kwargs['rvs']['rvs'], obs_d, params)
            if out is None:
                rvr, u = self._rvs_device(kwargs)
                out = K.flps_sv_corr(obs_d, torch.from_numpy(params).to(self.device), rvr, u,
                                     lag=self.settings['fixed_lag'], compute_hessian=hessian_flag,
                                     ctas_per_problem=self.ctas_per_problem, workspace=self._workspace)
            xf, xs, ll, grad, xtraj, hess1, hess2, diag = self._to_host(
                [out['filt'][0], out['smo'][0], out['log_like'], out['gradient'][0], out['traj'][0],
                 out['hess1'][0], out['hess2'][0], out['diag'][0]])
            return self._publish_smoother(model, xf, xs, ll, grad, xtraj, hess1, hess2, diag)
        except Exception as e:
            print("Error in CUDA code for particle smoother.")
            print(e)
            return False

    def _publish_smoother(self, model, xf, xs, ll, grad, xtraj, hess1, hess2, diag):
        """Host arrays of one evaluation -> `results` (cython.py:100-126); raises on a degenerate cloud."""
        self.diagnostics = {'near_ties': int(diag[DIAG_NEAR_TIES]), 'status': int(diag[DIAG_STATUS])}
        if int(diag[DIAG_STATUS]) != 0:
            raise FloatingPointError("degenerate particle cloud")

        # estimate of gradient and Hessian, cython.py:100-114 (Q9: np.inner is a scalar)
        if model.using_gradients or model.using_hessians:
            grad = np.array(grad).reshape((model.no_params, model.no_obs + 1))
            grad[np.isinf(grad)] = 0.0
            grad[np.isnan(grad)] = 0.0
            grad_est = np.nansum(grad, axis=1)
        if model.using_hessians and self.pairing == 'exact':
            hessian_est = np.outer(grad_est, grad_est) - (np.array(hess1).reshape((model.no_params, model.no_params)) +
                                                          np.array(hess2).reshape((model.no_params, model.no_params)))
        elif model.using_hessians:
            part1 = np.inner(grad_est, grad_est)
            part2 = np.array(hess1).reshape((model.no_params, model.no_params))
            part2 += np.array(hess2).reshape((model.no_params, model.no_params))
            hessian_est = part1 - part2

        self.results.update({'filt_state_est': np.array(xf).flatten()})
        self.results.update({'state_trajectory': np.array(xtraj).flatten()})
        self.results.update({'smo_state_est': np.array(xs).flatten()})
        self.results.update({'log_like': float(np.asarray(ll).reshape(-1)[0])})
        if model.using_gradients or model.using_hessians:
            self.results.update({'log_joint_gradient_estimate': grad_est})
        if model.using_hessians:
            self.results.update({'log_joint_hessian_estimate': -hessian_est})
        if self._estimate_gradient_and_hessian(model):
            return True
        return False

    # -------------------------------------------------------------------- init
    def _init_particle_method(self, model, no_particles, fixed_lag, verbose):
        no_obs = model.no_obs + 1
        self.name = "Particle method (CUDA) for " + model.short_name + " model"
        self.alg_type = 'particle'
        self.settings = {'no_particles': no_particles,
                         'no_obs': no_obs,
                         'resampling_method': 'systematic',
                         'fixed_lag': fixed_lag,
                         'initial_state': 0.0,
                         'generate_initial_state': True,
                         'estimate_gradient': True,
                         'estimate_hessian': True,
                         'pairing': self.pairing
                         }
        self.no_obs = no_obs
        self.no_particles = no_particles
        self.dim_rvs = (no_obs, no_particles + 1)
        if verbose:
            print("CUDA particle smoothing implementation for " + model.short_name + " initialised.")
            for key in self.settings:
                print("{}: {}".format(key, self.settings[key]))
