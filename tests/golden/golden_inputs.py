"""Seeded input generators shared by tests/golden/make_golden.py and the tests.

NumPy only (``RandomState`` streams are reproducible across machines), so the golden
files need to store outputs, not inputs.  Shapes follow BASELINE.json / SURVEY.md
section 8(d); layouts follow the reference:

* ``rvs`` for the particle estimators has shape (NOBS, N+1); the reference flattens it and
  splits it FLAT: ``rv_r = Phi(flat[:NOBS])``, ``rv_p = flat[NOBS:]`` with kernel index
  ``rvp[i + j*NOBS]`` (state/particle_methods/cython.py:89-91).
* the importance sampler uses ``rv_r = Phi(rvs[0, 0])``, ``rv_p = rvs[:, 1:].flatten()``
  (state/importance_sampling/cython.py:82-83).
"""
import numpy as np
from scipy.stats import norm

# (N, NOBS, LAG, seeds)
SV_KERNEL_CASES = [
    (75, 361, 10, (0, 1, 2)),      # shipped constants
    (37, 50, 10, (0, 1)),          # N < NOBS
    (200, 120, 10, (0, 1)),        # N > NOBS: Q7 / Q10 reach slots > 0
    (64, 40, 4, (0, 1)),           # other LAG
    (1024, 1001, 10, (0,)),        # BASELINE config 2, smallest N
    (4096, 1001, 10, (0,)),        # BASELINE config 4 per-chain size
]
RE_KERNEL_CASES = [(100, 100, (0, 1, 2)), (64, 37, (0, 1))]
SS_KERNEL_CASES = [(5500, 110000, (0, 1)), (77, 1000, (0, 1, 2))]

SV_PARAM_SETS = [
    (0.2, 0.9, 0.4, -0.5),    # data-generating values (SURVEY 8d)
    (2.0, 0.9, 0.4, -0.2),    # the paper's MH start, example3_stochastic_volatility.py:27
    (-0.3, 0.97, 0.15, 0.3),
]
SV_ESTIMATOR_PARAMS = [(0.2, 0.9, 0.4, -0.5), (2.0, 0.9, 0.4, -0.2)]
RE_ESTIMATOR_PARAMS = [(1.0, 0.2), (0.7, 0.35)]
LOGIT_D = 22


def sv_obs(nobs, params=(0.2, 0.9, 0.4, -0.5), seed=87655678):
    """Synthetic returns from the SV-with-leverage model
    (models/stochastic_volatility.py:32-37), length NOBS = T+1."""
    mu, phi, sigmav, rho = params
    rs = np.random.RandomState(seed)
    n = int(nobs)
    x = mu + sigmav / np.sqrt(1.0 - phi * phi) * rs.normal()
    y = np.zeros(n)
    for t in range(n):
        e = rs.normal()
        v = rho * e + np.sqrt(1.0 - rho * rho) * rs.normal()
        y[t] = np.exp(0.5 * x) * e
        x = mu + phi * (x - mu) + sigmav * v
    return y


def sv_rvs(n, nobs, seed):
    return np.random.RandomState(seed).normal(size=(nobs, n + 1))


def split_particle(rvs, nobs):
    flat = np.asarray(rvs, dtype=np.float64).flatten()
    return norm.cdf(flat[0:nobs]).flatten(), np.ascontiguousarray(flat[nobs:])


def sv_inputs(n, nobs, seed):
    """(obs[NOBS], params[4], rvr[NOBS], rvp[NOBS*N]) for kernel-level cases."""
    obs = sv_obs(nobs)
    params = np.array(SV_PARAM_SETS[seed % len(SV_PARAM_SETS)], dtype=np.float64)
    rvr, rvp = split_particle(sv_rvs(n, nobs, seed), nobs)
    return obs, params, rvr, rvp


def re_obs(nobs, mu=1.0, sigma=0.2, seed=87655678):
    """Random-effects data: x_i ~ N(mu, sigma^2), y_i ~ N(x_i, 1)
    (scripts/helper_random_effects.py:36-40)."""
    rs = np.random.RandomState(seed)
    x = mu + sigma * rs.normal(size=nobs)
    return x + rs.normal(size=nobs)


def re_rvs(n, nobs, seed):
    return np.random.RandomState(seed).normal(size=(nobs, n + 1))


def re_inputs(n, nobs, seed):
    obs = re_obs(nobs)
    params = np.array(RE_ESTIMATOR_PARAMS[seed % len(RE_ESTIMATOR_PARAMS)], dtype=np.float64)
    rvs = re_rvs(n, nobs, seed)
    rvr = float(norm.cdf(rvs[:, 0][0]))
    rvp = np.ascontiguousarray(rvs[:, 1:].flatten())
    return obs, params, rvr, rvp


def ss_inputs(m, seed):
    """Sorted uniforms as state/direct/standard.py:75 builds them."""
    u = np.random.RandomState(seed).normal(size=m)
    return np.sort(norm.cdf(u))


def logit_data(n, d, seed=0):
    """Higgs-shaped synthetic logistic data (SURVEY 8d config 3)."""
    rs = np.random.RandomState(seed)
    x = rs.normal(size=(n, d))
    beta = 0.1 * rs.normal(size=d)
    p = 1.0 / (1.0 + np.exp(-x.dot(beta)))
    y = (rs.uniform(size=n) < p).astype(np.float64)
    return x, y, beta


def logit_prior(d):
    return None


def logit_u(m, seed):
    return np.random.RandomState(seed).normal(size=m)


# phi = 0: the propagation mean is 0 for every parent, so the predicted child range collapses to +- nsd sd
LG_PARAM_SETS = [(0.8, 0.5, 0.3, 0.0), (0.95, 0.2, 1.0, 0.0), (-0.5, 1.0, 0.5, 0.0), (0.0, 0.7, 0.5, 0.0)]


def lg_obs(nobs, params=(0.8, 0.5, 0.3, 0.0), seed=4711):
    """Synthetic data from x' = phi x + sigma_v v, y = x + sigma_e e, x_0 = 0 (csrc/pf_model.cuh)."""
    phi, sv, se = params[:3]
    rs = np.random.RandomState(seed)
    x, y = 0.0, np.zeros(int(nobs))
    for t in range(1, int(nobs)):
        x = phi * x + sv * rs.normal()
        y[t] = x + se * rs.normal()
    return y


def lg_inputs(n, nobs, seed):
    params = np.array(LG_PARAM_SETS[seed % len(LG_PARAM_SETS)], dtype=np.float64)
    obs = lg_obs(nobs, params)
    rvr, rvp = split_particle(sv_rvs(n, nobs, 100 + seed), nobs)
    return obs, params, rvr, rvp
