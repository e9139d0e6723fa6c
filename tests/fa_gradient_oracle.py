"""TEST INFRASTRUCTURE ONLY -- the restatement and the exact targets of model id 4 (csrc/pf_model.cuh
LinearGaussianFullyAdaptedGrad: model 2's fully adapted linear Gaussian filter with a fixed-lag gradient under the
predictive pairing, kPredictiveScore).  Nothing under pmmh-qn_b200/ imports it.

Restatement.  Model 4's particle system is model 2's, so flps_fa_grad runs model 2's restatement
(oracle/generic_pf.py flps_generic with LinearGaussianFullyAdapted) for filt, smo, log_like, traj and the history
(X, A, W), and replays that history operation for operation the way flps_generic carries the lagged ancestors (ph) to
add the gradient: at step i >= L - 1 the pair (x_tt, x_tt+1), tt = i - L + 1, with y = obs[tt] under W_i into slot tt;
in the tail t = NOBS-L+1 .. NOBS-1 the pair (x_t, x_t+1) with y = obs[t] under W_{NOBS-1} into slot t, and for
t = NOBS-1 the final term score_last(x_{NOBS-1}, obs[NOBS-1]) under W_{NOBS-1}.

Exact targets (fa_gradient_targets, on oracle/kalman.py's filter and RTS moments; the kernel runs on obs[1:], T' = T - 1
slots): slot k <= T' - 2 is pair_score of (x_k, x_{k+1}) with y_{k+1} given y_{1:c(k)+1}, c(k) = min(k + L - 1, T' - 1);
slot T' - 1 = T - 2 is the predictive score grad log N(y_{T-1}; phi x_{T-2}, sigma_v^2 + sigma_e^2) given y_{1:T-1}.
The slots sum to the score of the full log-likelihood.
"""
import numpy as np

import generic_pf as gp
import kalman as km


class LinearGaussianFullyAdaptedGrad(gp.LinearGaussianFullyAdapted):
    """csrc/pf_model.cuh LinearGaussianFullyAdaptedGrad's score terms, operation for operation (precomputed reciprocals)."""

    def __init__(self, params):
        gp.LinearGaussianFullyAdapted.__init__(self, params)
        self.inv_sv2 = 1.0 / (self.sv * self.sv)
        self.inv_sv = 1.0 / self.sv
        self.inv_se2 = 1.0 / (self.se * self.se)
        self.inv_se = 1.0 / self.se

    def score_main(self, curr, nxt, y):
        """d/d(phi, sigma_v, sigma_e) of log N(nxt; phi curr, sigma_v^2) + log N(y; nxt, sigma_e^2)"""
        r = nxt - self.phi * curr
        ry = y - nxt
        g0 = (r * curr) * self.inv_sv2
        g1 = ((r * r) * self.inv_sv2 - 1.0) * self.inv_sv
        g2 = ((ry * ry) * self.inv_se2 - 1.0) * self.inv_se
        return np.stack([g0, g1, g2, np.zeros_like(g0)])

    score_tail = score_main

    def score_last(self, x, y_next):
        """d/d(phi, sigma_v, sigma_e) of log N(y_next; phi x, sigma_v^2 + sigma_e^2)"""
        r = y_next - self.phi * x
        a = (r * r) * self.inv_s2 - 1.0
        g0 = (r * x) * self.inv_s2
        g1 = (a * self.sv) * self.inv_s2
        g2 = (a * self.se) * self.inv_s2
        return np.stack([g0, g1, g2, np.zeros_like(g0)])


def predictive_gradient(model, obs, X, A, W, lag):
    """gradient [4][NOBS] of the predictive pairing from a run's history (X, A, W sorted by generation)."""
    obs = np.asarray(obs, dtype=np.float64)
    nobs, n, L = X.shape[0], X.shape[1], int(lag)
    grad = np.zeros((4, nobs))
    ph = np.zeros((L, n))                                          # ph[k][j]: ancestor k steps back of particle j
    ph[0] = X[0]
    for i in range(1, nobs):
        oph = ph.copy()
        ph[0] = X[i]
        ph[1:] = oph[:-1][:, A[i]]
        if i >= L - 1:
            tt = i - L + 1
            grad[:, tt] += np.sum(model.score_main(ph[L - 1], ph[L - 2], obs[tt]) * W[i], axis=1)
    for t in range(nobs - L + 1, nobs):                            # tail: final weights
        k = nobs - 1 - t
        if k >= 1:
            grad[:, t] += np.sum(model.score_tail(ph[k], ph[k - 1], obs[t]) * W[nobs - 1], axis=1)
        else:
            grad[:, t] += np.sum(model.score_last(ph[0], obs[t]) * W[nobs - 1], axis=1)
    return grad


def flps_fa_grad(params, obs, rvr, rvp, n_particles, lag=10, dumps=False):
    """Model 4 on the shifted series obs (= the full series [1:]): flps_generic's outputs of model 2 with the gradient of
    the predictive pairing."""
    out = gp.flps_generic(gp.LinearGaussianFullyAdapted(params), obs, rvr, rvp, n_particles, lag, dumps=True)
    out["gradient"] = predictive_gradient(LinearGaussianFullyAdaptedGrad(params), obs, out["X"], out["A"], out["W"], lag)
    if not dumps:
        for k in ("X", "A", "W"):
            del out[k]
    return out


def predictive_score(phi, sv, se, m, p, y):
    """E[grad log N(y; phi x, sv^2 + se^2)] over (phi, sv, se) for x ~ N(m, p)."""
    s2 = sv * sv + se * se
    erx = y * m - phi * (p + m * m)                    # E[(y - phi x) x]
    er2 = (y - phi * m) ** 2 + phi * phi * p           # E[(y - phi x)^2]
    a = er2 / s2 - 1.0
    return np.array([erx / s2, a * sv / s2, a * se / s2])


def fa_gradient_targets(obs, phi, sv, se, lag):
    """Exact targets of model 4's gradient for the full series obs (the kernel runs on obs[1:]): grad[3][T - 1] per slot,
    grad_sum[3], and mom[k] = (c, moments) the targets were computed from (the last entry (T - 1, m, p))."""
    obs = np.asarray(obs, dtype=np.float64)
    T = obs.shape[0]
    n = T - 1
    kf = km.kalman_filter(obs, phi, sv, se)
    grad = np.zeros((3, n))
    mom = []
    for k in range(n - 1):
        c = km.conditioning_index(k, lag, n, 1)
        ms, ps, cs = km.rts(kf, c, k, phi)
        grad[:, k] = km.pair_score(phi, sv, se, ms[0], ps[0], ms[1], ps[1], cs[0], obs[k + 1])
        mom.append((c, ms[0], ps[0], ms[1], ps[1], cs[0]))
    ms, ps, _ = km.rts(kf, T - 1, T - 2, phi)
    grad[:, n - 1] = predictive_score(phi, sv, se, ms[0], ps[0], obs[T - 1])
    mom.append((T - 1, ms[0], ps[0]))
    return dict(grad=grad, grad_sum=grad.sum(axis=1), mom=mom)
