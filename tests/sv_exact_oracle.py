"""TEST INFRASTRUCTURE ONLY -- the restatement of model id 8 (csrc/pf_model.cuh SvLeverageExact: the SV model's
particle system with the exact fixed-lag score and the generic Hessian branch).  Nothing under pmmh-qn_b200/ imports it.

Model 8's particle system is model 0's, so flps_sv_exact runs oracle/generic_pf.py's flps_generic with
SvLeverageExact (model 0's propagation and weights; reference_indexing False gives the smo of the exact pairings) and
replays that history with predictive_replay: at step i >= L - 1 the pair (x_tt, x_tt+1), tt = i - L + 1, with
y = obs[tt] under W_i into slot tt (the pair (x_0, x_1) through score_first / hess_first), in the tail
t = NOBS-L+1 .. NOBS-2 the pair (x_t, x_t+1) under W_{NOBS-1} into slot t, and score_last (0 here) into slot NOBS-1.
The Hessian carries alpha along every lineage as tests/fa_hessian_oracle.py describes.  predictive_replay takes any model
with the hooks: on models 4 and 6 it reproduces tests/fa_gradient_oracle.predictive_gradient and
tests/fa_hessian_oracle.predictive_hessian, which have no first-pair hook (test_sv_exact_reference.py).

Parameters: theta = (mu, atanh phi, log sigma_v, atanh rho), the reference's free parametrisation; hooks in closed form
(derivation in csrc/pf_model.cuh).
"""
import numpy as np

import generic_pf as gp
from fa_hessian_oracle import _terms


def _sym(v):
    """the 4 x 4 symmetric matrices of 10 upper-triangle entries (row by row) [10][...] -> [4][4][...]"""
    v = [np.asarray(e, dtype=np.float64) for e in v]
    shape = np.broadcast(*v).shape
    out = np.zeros((4, 4) + shape)
    z = 0
    for i in range(4):
        for j in range(i, 4):
            out[i, j] = out[j, i] = v[z]
            z += 1
    return out


class SvLeverageExact(gp.SvLeverage):
    """csrc/pf_model.cuh SvLeverageExact's hooks: score_main is model 0's (stochastic_volatility.pyx:452-465 with the
    pair's own observation), score_tail the same, score_last 0; hooks on arrays of particles."""
    reference_indexing = False

    def __init__(self, params):
        gp.SvLeverage.__init__(self, params)

    @classmethod
    def from_theta(cls, theta):
        mu, a, b, c = [float(v) for v in theta]
        return cls((mu, np.tanh(a), np.exp(b), np.tanh(c)))

    def trans_sd(self):
        return np.sqrt(self.rho_term) * self.sv

    def score_tail(self, curr, nxt, y):
        return self.score_main(curr, nxt, y)

    def score_last(self, x, y_next):
        return np.zeros((4,) + np.shape(x))

    def score_first(self, x1, y0):
        x1 = np.asarray(x1, dtype=np.float64)
        g = self.score_main(np.full_like(x1, self.mu), x1, y0)
        ey = np.exp(-0.5 * self.mu) * y0
        sq = x1 - self.mu - self.sv * self.rho * ey
        g[0] = self.q * sq * (1.0 - 0.5 * self.sv * self.rho * ey)
        g[1] = 0.0
        return g

    def _hess(self, s, ds, d2s):
        """second derivatives of 1/2 log q - q s^2 / 2 from s and its derivatives (ds [4], d2s [10] upper triangle)"""
        dlq = (0.0, 0.0, -2.0, 2.0 * self.rho)
        h, z = [], 0
        for i in range(4):
            for j in range(i, 4):
                v = (-0.5 * self.q * s * s * dlq[i] * dlq[j] - self.q * s * (dlq[i] * ds[j] + ds[i] * dlq[j])
                     - self.q * ds[i] * ds[j] - self.q * s * d2s[z])
                if i == 3 and j == 3:
                    v = v + self.rho_term * (1.0 - self.q * s * s)
                h.append(v)
                z += 1
        return _sym(h)

    def hess_main(self, curr, nxt, y):
        curr, nxt = np.asarray(curr, dtype=np.float64), np.asarray(nxt, dtype=np.float64)
        d, ey, p, r = curr - self.mu, np.exp(-0.5 * curr) * y, 1.0 - self.phi ** 2, self.rho_term
        sr = self.sv * self.rho
        s = nxt - self.mu - self.phi * d - sr * ey
        ds = (-(1.0 - self.phi), -d * p, -sr * ey, -self.sv * ey * r)
        d2s = (0.0, p, 0.0, 0.0, 2.0 * self.phi * p * d, 0.0, 0.0, -sr * ey, -self.sv * ey * r, 2.0 * sr * ey * r)
        return self._hess(s, ds, d2s)

    def hess_first(self, x1, y0):
        x1 = np.asarray(x1, dtype=np.float64)
        ey, r, sr = np.exp(-0.5 * self.mu) * y0, self.rho_term, self.sv * self.rho
        s = x1 - self.mu - sr * ey
        ds = (-(1.0 - 0.5 * sr * ey), 0.0, -sr * ey, -self.sv * ey * r)
        d2s = (-0.25 * sr * ey, 0.0, 0.5 * sr * ey, 0.5 * self.sv * ey * r, 0.0, 0.0, 0.0, -sr * ey,
               -self.sv * ey * r, 2.0 * sr * ey * r)
        return self._hess(s, ds, d2s)

    def hess_last(self, x, y_next):
        return np.zeros((4, 4) + np.shape(x))

    def trans_logpdf(self, curr, nxt, y):
        """log N(nxt; mu + phi (curr - mu) + sigma_v rho e^{-curr/2} y, sigma_v^2 (1 - rho^2))"""
        m = self.propagate(curr, y, 0.0)
        s2 = self.rho_term * self.sv * self.sv
        return -0.5 * np.log(2.0 * np.pi * s2) - 0.5 * (nxt - m) ** 2 / s2


def _pair(model, fn, first, curr, nxt, y):
    """score / hess of the pair (curr, nxt): the first-pair hook where the model has one"""
    if first and hasattr(model, fn + "_first"):
        return getattr(model, fn + "_first")(nxt, y)
    return getattr(model, fn + "_main")(curr, nxt, y)


def predictive_replay(model, obs, X, A, W, lag, hessian=False):
    """gradient [4][NOBS] of the predictive pairing from a run's history (X, A, W sorted by generation), and with
    `hessian` (hess1, hess2) [4][4] by Louis' identity (alpha(x_0) = 0, alpha(child) = alpha(parent) + the pair's
    score at the child's birth)."""
    obs = np.asarray(obs, dtype=np.float64)
    nobs, n, L = X.shape[0], X.shape[1], int(lag)
    grad = np.zeros((4, nobs))
    h1, h2 = np.zeros((4, 4)), np.zeros((4, 4))
    ph = np.zeros((L, n))          # ph[k][j]: value of the ancestor k steps back of particle j
    pa = np.zeros((L, 4, n))       # pa[k][:, j]: its alpha
    ph[0] = X[0]
    for i in range(1, nobs):
        oph, opa = ph.copy(), pa.copy()
        ph[0] = X[i]
        ph[1:] = oph[:-1][:, A[i]]
        if hessian:
            pa[1:] = opa[:-1][:, :, A[i]]
            pa[0] = pa[1] + _pair(model, "score", i == 1, ph[1], ph[0], obs[i - 1])
        if i >= L - 1:
            tt = i - L + 1
            curr, nxt = ph[L - 1], ph[L - 2]
            s = _pair(model, "score", tt == 0, curr, nxt, obs[tt])
            grad[:, tt] += np.sum(s * W[i], axis=1)
            if hessian:
                a1, a2 = _terms(s, _pair(model, "hess", tt == 0, curr, nxt, obs[tt]), pa[L - 1], W[i])
                h1 += a1
                h2 += a2
    for t in range(nobs - L + 1, nobs):                            # tail: final weights
        k = nobs - 1 - t
        if k >= 1:
            s = model.score_tail(ph[k], ph[k - 1], obs[t])
            h = model.hess_main(ph[k], ph[k - 1], obs[t]) if hessian else None
        else:
            s = model.score_last(ph[0], obs[t])
            h = model.hess_last(ph[0], obs[t]) if hessian else None
        grad[:, t] += np.sum(s * W[nobs - 1], axis=1)
        if hessian:
            a1, a2 = _terms(s, h, pa[k], W[nobs - 1])
            h1 += a1
            h2 += a2
    return (grad, h1, h2) if hessian else grad


def flps_sv_exact(params, obs, rvr, rvp, n_particles, lag=10, dumps=False, hessian=False):
    """Model 8: flps_generic's filt, smo, log_like, traj (model 0's particle system) with the gradient of the predictive
    pairing, and hess1 / hess2 [4][4] with `hessian`."""
    model = SvLeverageExact(params)
    out = gp.flps_generic(model, obs, rvr, rvp, n_particles, lag, dumps=True)
    r = predictive_replay(model, obs, out["X"], out["A"], out["W"], lag, hessian)
    if hessian:
        out["gradient"], out["hess1"], out["hess2"] = r
    else:
        out["gradient"] = r
    if not dumps:
        for k in ("X", "A", "W"):
            del out[k]
    return out


def hessian_estimate(out):
    """hess1 + hess2 - g g' over theta, g = the summed gradient slots"""
    g = np.asarray(out["gradient"]).sum(axis=1)
    return np.asarray(out["hess1"]) + np.asarray(out["hess2"]) - np.outer(g, g)
