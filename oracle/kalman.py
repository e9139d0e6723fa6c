"""TEST INFRASTRUCTURE ONLY -- exact fp64 Kalman quantities of the linear Gaussian model that the particle
smoother's outputs estimate (csrc/pf_model.cuh, model ids 1 and 2; oracle/generic_pf.py restates the kernels).

Model and convention (generic_pf.kalman_loglike's): x_0 = 0 fixed, x_t = phi x_{t-1} + sigma_v v_t,
y_t = obs[t] = x_t + sigma_e e_t for t = 1 .. T-1 (T = len(obs)); obs[0] is not weighted.

What the estimators target (exact pairing, generic_pf.flps_generic with reference_indexing False):
  * model 1 `filt[t]` = E[x_t | y_{1:t}];
  * model 2 runs on obs[1:] and weights generation t with p(y_{t+1} | x_t): `filt[t]` = E[x_t | y_{1:t+1}];
  * `smo[t]` is read under the weights of generation c(t) = min(t + L - 1, T' - 1) (T' = the length of the series the
    kernel sees): E[x_t | y_{1:c(t)}] for model 1 and E[x_t | y_{1:c(t)+1}] for model 2;
  * gradient slot s = t + 1 holds E[score of the pair (x_t, x_{t+1}) | y_{1:c(t)}] (model 1), where the pair's score is
    grad log N(x_{t+1}; phi x_t, sigma_v^2) + grad log N(y_{t+1}; x_{t+1}, sigma_e^2) over (phi, sigma_v, sigma_e);
    slot 0 is 0.
Each conditional expectation is an RTS pass over exactly the observations its estimator conditions on, with the lag-one
cross-covariance Cov(x_t, x_{t+1} | y_{1:c}) = J_t P_{t+1|c}.  So no lag-truncation allowance enters a comparison.
"""
import numpy as np


def kalman_filter(obs, phi, sv, se):
    """Filtered and one-step predicted moments: m[t] = E[x_t | y_{1:t}], p[t] = Var, mp[t] / pp[t] = the same given
    y_{1:t-1} (t >= 1); index 0 is x_0 = 0 (variance 0)."""
    y = np.asarray(obs, dtype=np.float64)
    T = y.shape[0]
    m, p, mp, pp = np.zeros(T), np.zeros(T), np.zeros(T), np.zeros(T)
    for t in range(1, T):
        mp[t], pp[t] = phi * m[t - 1], phi * phi * p[t - 1] + sv * sv
        k = pp[t] / (pp[t] + se * se)
        m[t], p[t] = mp[t] + k * (y[t] - mp[t]), (1.0 - k) * pp[t]
    return m, p, mp, pp


def rts(kf, c, t0, phi):
    """Moments of x_{t0 .. c} given y_{1:c} by the RTS recursion from c down to t0 over the filter `kf`:
    (mean, var, cross) with cross[t - t0] = Cov(x_t, x_{t+1} | y_{1:c}) (last entry 0)."""
    m, p, mp, pp = kf
    n = c - t0 + 1
    ms, ps, cs = np.zeros(n), np.zeros(n), np.zeros(n)
    ms[-1], ps[-1] = m[c], p[c]
    for t in range(c - 1, t0 - 1, -1):
        j = p[t] * phi / pp[t + 1]                     # J_t (0 at t = 0: x_0 is fixed)
        k = t - t0
        ms[k] = m[t] + j * (ms[k + 1] - mp[t + 1])
        ps[k] = p[t] + j * j * (ps[k + 1] - pp[t + 1])
        cs[k] = j * ps[k + 1]
    return ms, ps, cs


def pair_score(phi, sv, se, m0, p0, m1, p1, c01, y1):
    """E[grad log N(x1; phi x0, sv^2) + grad log N(y1; x1, se^2)] over (phi, sv, se) for (x0, x1) Gaussian with means
    m0, m1, variances p0, p1 and covariance c01."""
    e00, e11, e01 = p0 + m0 * m0, p1 + m1 * m1, c01 + m0 * m1
    er_x0 = e01 - phi * e00                            # E[(x1 - phi x0) x0]
    er2 = e11 - 2.0 * phi * e01 + phi * phi * e00      # E[(x1 - phi x0)^2]
    ery2 = (y1 - m1) ** 2 + p1                         # E[(y1 - x1)^2]
    return np.array([er_x0 / (sv * sv), (er2 / (sv * sv) - 1.0) / sv, (ery2 / (se * se) - 1.0) / se])


def filtered_means(obs, phi, sv, se):
    """Model 1's `filt`: E[x_t | y_{1:t}]."""
    return kalman_filter(obs, phi, sv, se)[0].copy()


def fa_filtered_means(obs, phi, sv, se):
    """Model 2's `filt` of a run on obs[1:] (length T - 1): E[x_t | y_{1:t+1}], a one-step smoother."""
    kf = kalman_filter(obs, phi, sv, se)
    T = len(obs)
    out = np.zeros(T - 1)
    for t in range(1, T - 1):
        out[t] = rts(kf, t + 1, t, phi)[0][0]
    return out


def conditioning_index(t, lag, n_kernel, shift=0):
    """Last observation the smoother's slot t conditions on: c(t) + shift, c(t) = min(t + lag - 1, n_kernel - 1)."""
    return min(t + lag - 1, n_kernel - 1) + shift


def fixed_lag_targets(obs, phi, sv, se, lag, fully_adapted=False):
    """Exact targets of the fixed-lag smoother's outputs.  Model 1 (fully_adapted False): smo[T], grad[3][T] per slot
    (slot 0 = 0) and grad_sum[3].  Model 2 (True, the kernel runs on obs[1:]): smo[T - 1]; no gradient.
    Also returns the moments every target was computed from: mom[t] = (c, m_t, p_t, m_{t+1}, p_{t+1}, cov)."""
    obs = np.asarray(obs, dtype=np.float64)
    T = obs.shape[0]
    kf = kalman_filter(obs, phi, sv, se)
    shift = 1 if fully_adapted else 0
    n = T - shift
    smo = np.zeros(n)
    grad = np.zeros((3, n))
    mom = []
    for t in range(n):
        c = conditioning_index(t, lag, n, shift)
        ms, ps, cs = rts(kf, c, t, phi)
        smo[t] = ms[0]
        if not fully_adapted and t + 1 < n:
            grad[:, t + 1] = pair_score(phi, sv, se, ms[0], ps[0], ms[1], ps[1], cs[0], obs[t + 1])
            mom.append((c, ms[0], ps[0], ms[1], ps[1], cs[0]))
    out = dict(smo=smo, mom=mom)
    if not fully_adapted:
        out.update(grad=grad, grad_sum=grad.sum(axis=1))
    return out
