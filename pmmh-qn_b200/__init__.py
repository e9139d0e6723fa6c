"""pmmh-qn_b200 -- B200 (sm_100a) implementation of the likelihood-estimation hot path of
compops/pmmh-qn: SV particle filter / fixed-lag smoother with sorted correlated systematic
resampling, the random-effects correlated importance sampler, the data-subsampling
estimator and the Crank-Nicolson update of the auxiliary variables u.

Layout
  csrc/     hand-written CUDA kernels + the extern "C" boundary (include/pmmh_qn.h)
  _lib.py   ctypes loader (fails loudly when the library is missing; no CPU fallback)
  kernels.py  torch-tensor wrappers (PyTorch = allocator and stream owner only)
  state/    host-side mirrors of the reference's estimator classes
            (ParticleMethodsCUDA, ImportanceSamplingCUDA, DirectComputationCUDA)
  parameter/  device-resident u handles and the Crank-Nicolson proposal
"""
__version__ = "0.1.0"

_LAZY = {
    "ParticleMethodsCUDA": ("state.particle_methods.cuda", "ParticleMethodsCUDA"),
    "ImportanceSamplingCUDA": ("state.importance_sampling.cuda", "ImportanceSamplingCUDA"),
    "DirectComputationCUDA": ("state.direct.cuda", "DirectComputationCUDA"),
    "LinearGaussianParticleMethodsCUDA": ("state.particle_methods.linear_gaussian", "LinearGaussianParticleMethodsCUDA"),
    "DeviceRVS": ("parameter.rvs", "DeviceRVS"),
    "propose_rvs": ("parameter.rvs", "propose_rvs"),
    "CorrelatedRVSState": ("parameter.rvs", "CorrelatedRVSState"),
}


def __getattr__(name):
    if name in _LAZY:
        import importlib
        mod, attr = _LAZY[name]
        return getattr(importlib.import_module(__name__ + "." + mod), attr)
    raise AttributeError(name)


def build(force=False, verbose=False):
    """Compile libpmmh_qn_b200.so in-tree (nvcc, sm_100a)."""
    from . import _build
    return _build.build(force=force, verbose=verbose)
