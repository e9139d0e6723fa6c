"""TEST INFRASTRUCTURE ONLY -- the restatement and the exact targets of model id 6 (csrc/pf_model.cuh
LinearGaussianFullyAdaptedHess: model 4 with the generic Hessian branch of the grid kernel).  Nothing under
pmmh-qn_b200/ imports it.

Restatement.  Model 6's particle system and gradient are model 4's, so flps_fa_hess runs tests/fa_gradient_oracle.py's
flps_fa_grad and replays model 2's history (X, A, W) the way predictive_gradient does, carrying with every lagged
ancestor value (ph) its alpha (pa): alpha(x_0) = 0 and alpha(child) = alpha(parent) + score_main(parent, child,
obs[i - 1]) at its birth (generation i).  Slot k's pair (x_k, x_k+1), read under the weights of generation c(k), adds
H_k = hess_main to hess1 and s_k s_k' + alpha_k s_k' + s_k alpha_k' to hess2, alpha_k = the alpha of x_k on the lineage
read; the final generation adds hess_last and the same hess2 term with its own alpha.  `mutation` changes one line:
  'alpha_own'   alpha_k + s_k (the pair's own term counted twice),
  'alpha_read'  the alpha of the particle at generation c(k) (alpha taken from the wrong generation),
  'drop_last'   the final generation's term missing.

Exact targets.  hess1_targets: E[H_k | y_1 .. y_c(k)+1] per slot from the RTS moments (H_k is linear in the first and
second moments of the pair); kalman_hessian: the Hessian of generic_pf.kalman_loglike over (phi, sigma_v, sigma_e) by
central differences.
"""
import numpy as np

import fa_gradient_oracle as fo
import generic_pf as gp
import kalman as km


def _sym(h00, h01, h02, h11, h12, h22):
    z = np.zeros_like(h00)
    return np.array([[h00, h01, h02, z], [h01, h11, h12, z], [h02, h12, h22, z], [z, z, z, z]])


class LinearGaussianFullyAdaptedHess(fo.LinearGaussianFullyAdaptedGrad):
    """csrc/pf_model.cuh LinearGaussianFullyAdaptedHess's Hessian hooks as full 4 x 4 matrices (per particle)."""

    def hess_main(self, curr, nxt, y):
        """second derivatives over (phi, sigma_v, sigma_e) of log N(nxt; phi curr, sigma_v^2) + log N(y; nxt, sigma_e^2)"""
        curr, nxt = np.asarray(curr, dtype=np.float64), np.asarray(nxt, dtype=np.float64)
        r = nxt - self.phi * curr
        ry = y - nxt
        z = np.zeros_like(r)
        return _sym(-(curr * curr) * self.inv_sv2, -2.0 * (r * curr) * (self.inv_sv2 * self.inv_sv), z,
                    (1.0 - 3.0 * (r * r) * self.inv_sv2) * self.inv_sv2, z,
                    (1.0 - 3.0 * (ry * ry) * self.inv_se2) * self.inv_se2)

    def hess_last(self, x, y_next):
        """second derivatives over (phi, sigma_v, sigma_e) of log N(y_next; phi x, sigma_v^2 + sigma_e^2)"""
        x = np.asarray(x, dtype=np.float64)
        r = y_next - self.phi * x
        a = (r * r) * self.inv_s2 - 1.0
        b = 2.0 * (r * r) * self.inv_s2 - 1.0
        i4 = self.inv_s2 * self.inv_s2
        return _sym(-(x * x) * self.inv_s2, -2.0 * (r * x) * self.sv * i4, -2.0 * (r * x) * self.se * i4,
                    (a - 2.0 * (self.sv * self.sv) * self.inv_s2 * b) * self.inv_s2, -2.0 * (self.sv * self.se) * i4 * b,
                    (a - 2.0 * (self.se * self.se) * self.inv_s2 * b) * self.inv_s2)


def _terms(s, h, al, w):
    """sum over particles of w H and w (s s' + al s' + s al'); s, al [4][n], h [4][4][n]"""
    h1 = np.sum(h * w, axis=2)
    h2 = np.einsum("an,bn,n->ab", s, s, w) + np.einsum("an,bn,n->ab", al, s, w) + np.einsum("an,bn,n->ab", s, al, w)
    return h1, h2


def predictive_hessian(model, obs, X, A, W, lag, mutation=None):
    """(hess1, hess2) [4][4] of model 6 from a run's history (X, A, W sorted by generation)."""
    obs = np.asarray(obs, dtype=np.float64)
    nobs, n, L = X.shape[0], X.shape[1], int(lag)
    h1, h2 = np.zeros((4, 4)), np.zeros((4, 4))
    ph = np.zeros((L, n))          # ph[k][j]: value of the ancestor k steps back of particle j
    pa = np.zeros((L, 4, n))       # pa[k][:, j]: its alpha
    ph[0] = X[0]
    for i in range(1, nobs):
        oph, opa = ph.copy(), pa.copy()
        ph[0] = X[i]
        ph[1:] = oph[:-1][:, A[i]]
        pa[1:] = opa[:-1][:, :, A[i]]
        pa[0] = pa[1] + model.score_main(ph[1], ph[0], obs[i - 1])
        if i >= L - 1:
            tt = i - L + 1
            curr, nxt = ph[L - 1], ph[L - 2]
            s = model.score_main(curr, nxt, obs[tt])
            al = {"alpha_own": pa[L - 1] + s, "alpha_read": pa[0]}.get(mutation, pa[L - 1])
            a1, a2 = _terms(s, model.hess_main(curr, nxt, obs[tt]), al, W[i])
            h1 += a1
            h2 += a2
    for t in range(nobs - L + 1, nobs):                            # tail: final weights
        k = nobs - 1 - t
        if k >= 1:
            s = model.score_tail(ph[k], ph[k - 1], obs[t])
            al = {"alpha_own": pa[k] + s, "alpha_read": pa[0]}.get(mutation, pa[k])
            a1, a2 = _terms(s, model.hess_main(ph[k], ph[k - 1], obs[t]), al, W[nobs - 1])
        elif mutation == "drop_last":
            continue
        else:
            s = model.score_last(ph[0], obs[t])
            al = pa[0] + s if mutation == "alpha_own" else pa[0]
            a1, a2 = _terms(s, model.hess_last(ph[0], obs[t]), al, W[nobs - 1])
        h1 += a1
        h2 += a2
    return h1, h2


def flps_fa_hess(params, obs, rvr, rvp, n_particles, lag=10, dumps=False, mutation=None):
    """Model 6 on the shifted series obs (= the full series [1:]): flps_fa_grad's outputs plus hess1 / hess2 [4][4]."""
    out = fo.flps_fa_grad(params, obs, rvr, rvp, n_particles, lag, dumps=True)
    out["hess1"], out["hess2"] = predictive_hessian(LinearGaussianFullyAdaptedHess(params), obs, out["X"], out["A"],
                                                    out["W"], lag, mutation)
    if not dumps:
        for k in ("X", "A", "W"):
            del out[k]
    return out


def hessian_estimate(out):
    """hess1 + hess2 - g g' over (phi, sigma_v, sigma_e), g = the summed gradient slots"""
    g = np.asarray(out["gradient"])[:3].sum(axis=1)
    return (np.asarray(out["hess1"]) + np.asarray(out["hess2"]))[:3, :3] - np.outer(g, g)


def hess1_targets(obs, phi, sv, se, lag):
    """Exact E[H_k | y_1 .. y_c(k)+1] [T - 1][3][3] per slot for the full series obs (the kernel runs on obs[1:]); the
    moments are fa_gradient_targets'."""
    obs = np.asarray(obs, dtype=np.float64)
    T = obs.shape[0]
    n = T - 1
    kf = km.kalman_filter(obs, phi, sv, se)
    out = np.zeros((n, 3, 3))
    for k in range(n - 1):
        c = km.conditioning_index(k, lag, n, 1)
        ms, ps, cs = km.rts(kf, c, k, phi)
        e00, e11, e01 = ps[0] + ms[0] ** 2, ps[1] + ms[1] ** 2, cs[0] + ms[0] * ms[1]
        erx = e01 - phi * e00
        er2 = e11 - 2.0 * phi * e01 + phi * phi * e00
        ery2 = (obs[k + 1] - ms[1]) ** 2 + ps[1]
        out[k] = _sym(-e00 / sv ** 2, -2.0 * erx / sv ** 3, 0.0, 1.0 / sv ** 2 - 3.0 * er2 / sv ** 4, 0.0,
                      1.0 / se ** 2 - 3.0 * ery2 / se ** 4)[:3, :3]
    ms, ps, _ = km.rts(kf, T - 1, T - 2, phi)
    m, p, y, s2 = ms[0], ps[0], obs[T - 1], sv * sv + se * se
    ex2, erx, er2 = p + m * m, y * m - phi * (p + m * m), (y - phi * m) ** 2 + phi * phi * p
    ea, eb = er2 / s2 - 1.0, 2.0 * er2 / s2 - 1.0
    out[n - 1] = _sym(-ex2 / s2, -2.0 * erx * sv / s2 ** 2, -2.0 * erx * se / s2 ** 2,
                      (ea - 2.0 * sv * sv / s2 * eb) / s2, -2.0 * sv * se / s2 ** 2 * eb,
                      (ea - 2.0 * se * se / s2 * eb) / s2)[:3, :3]
    return out


def kalman_hessian(obs, phi, sv, se, h=1e-4):
    """Hessian of generic_pf.kalman_loglike(obs) over (phi, sigma_v, sigma_e), central differences"""
    p0 = np.array([phi, sv, se], dtype=np.float64)
    f = lambda p: gp.kalman_loglike(obs, *p)
    out = np.zeros((3, 3))
    for a in range(3):
        for b in range(3):
            ea, eb = np.eye(3)[a] * h, np.eye(3)[b] * h
            out[a, b] = (f(p0 + ea + eb) - f(p0 + ea - eb) - f(p0 - ea + eb) + f(p0 - ea - eb)) / (4.0 * h * h)
    return 0.5 * (out + out.T)
