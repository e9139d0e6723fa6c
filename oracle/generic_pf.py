"""TEST INFRASTRUCTURE ONLY -- NumPy restatement of the reference's fixed-lag particle smoother
(/root/reference/python/state/particle_methods/stochastic_volatility.pyx:205-655, gradient branch) with
the model's three ingredients passed in as callbacks, the way python/README.md:73-76 describes porting
the Cython code to another scalar-state model.  It is the checker for the model-generic device entry
point pmmh_flps_model_corr (csrc/pf_model.cuh); nothing under pmmh-qn_b200/ imports it.

Pinning: with the SV callbacks below it must reproduce oracle_flps_sv_corr (oracle/pmmh_oracle.c, itself
bit-exact against the compiled reference) -- tests/test_oracle_vs_golden.py checks ancestors and sorted
generations exactly and the estimates to 1e-12 (NumPy's pairwise sums order the additions differently).
For the linear Gaussian model (bootstrap filter, model id 1, and fully adapted filter, model id 2) there is no
reference implementation, so there is no parity to keep: the fixed-lag terms pair the states exactly (no Q5 / Q6,
see flps_generic).  The device instantiations are pinned to the restatements below (ancestors exact), and the
restatements are pinned statistically to the exact fixed-lag Kalman quantities of oracle/kalman.py
(tests/test_kalman_reference.py).  The fully adapted restatement is itself checked against closed forms
(tests/test_oracle_vs_golden.py): its proposal against the precision-weighted conditional moments, its
likelihood estimate against the exact Kalman likelihood (statistically).
"""
import numpy as np


class SvLeverage(object):
    """stochastic_volatility.pyx:306-323 (Q1), :354-358, :427-437, :452-465, :548-557"""
    n_params = 4
    reference_indexing = True          # the reference's pairing of the fixed-lag terms (Q5 / Q6)

    def __init__(self, params):
        self.mu, self.phi, self.sv, self.rho = [float(p) for p in params]
        self.q = 1.0 / (self.sv * self.sv * (1.0 - self.rho * self.rho))
        self.rho_term = 1.0 - self.rho * self.rho

    def initial_state(self):
        return self.mu + (self.sv / np.sqrt(1.0 - self.phi * self.phi)) * 0.0

    def propagate(self, xp, y_prev, u):
        mean = self.mu + self.phi * (xp - self.mu)
        mean = mean + self.sv * self.rho * np.exp(-0.5 * xp) * y_prev
        return mean + np.sqrt(self.rho_term) * self.sv * u

    def logw(self, x, y):
        s = np.exp(0.5 * x)
        return -0.91893853320467267 + (-np.log(s)) + (-0.5 * (y - 0.0) * (y - 0.0) / (s * s))

    def score_main(self, curr, nxt, y):
        sq = nxt - self.mu - self.phi * (curr - self.mu)
        sq = sq - self.sv * self.rho * np.exp(-0.5 * curr) * y
        g0 = self.q * sq * (1.0 - self.phi)
        g1 = self.q * sq * (curr - self.mu) * (1.0 - self.phi ** 2.0)
        g2 = sq + self.sv * self.rho * np.exp(-0.5 * curr) * y
        g2 = g2 * (self.q * sq) - 1.0
        g3 = self.rho - self.q * self.rho * sq * sq
        g3 = g3 + self.sv ** -1.0 * sq * np.exp(-0.5 * curr) * y
        return np.stack([g0, g1, g2, g3])

    def score_tail(self, curr, nxt, y):
        sq = nxt - self.mu - self.phi * (curr - self.mu)
        sq = sq - self.sv * self.rho * np.exp(-0.5 * curr) * y
        g0 = self.q * sq * (1.0 - self.phi)
        g1 = self.q * sq * (curr - self.mu) * (1.0 - self.phi ** 2.0)
        g2 = self.q * sq * sq - 1.0 + self.q * sq * self.sv * self.rho * np.exp(-0.5 * curr) * y
        g3 = self.rho - self.q * self.rho * sq * sq + self.q * sq * self.sv * np.exp(-0.5 * curr) * y * self.rho_term
        return np.stack([g0, g1, g2, g3])


class LinearGaussian(object):
    """x' = phi x + sigma_v v, y = x + sigma_e e; params (phi, sigma_v, sigma_e, unused) -- csrc/pf_model.cuh"""
    n_params = 3
    reference_indexing = False         # exact pairing (flps_generic)

    def __init__(self, params):
        self.phi, self.sv, self.se = [float(p) for p in params[:3]]

    def initial_state(self):
        return 0.0

    def propagate(self, xp, y_prev, u):
        return self.phi * xp + self.sv * u

    def logw(self, x, y):
        r = y - x
        return (-0.91893853320467267 - np.log(self.se)) - (0.5 * (r * r)) / (self.se * self.se)

    def score_main(self, curr, nxt, y):
        """d/d(phi, sigma_v, sigma_e) of log N(nxt; phi curr, sigma_v^2) + log N(y; nxt, sigma_e^2), y = obs[time(nxt)]"""
        r = nxt - self.phi * curr
        ry = y - nxt
        g0 = (r * curr) / (self.sv * self.sv)
        g1 = ((r * r) / (self.sv * self.sv) - 1.0) / self.sv
        g2 = ((ry * ry) / (self.se * self.se) - 1.0) / self.se
        return np.stack([g0, g1, g2, np.zeros_like(g0)])

    score_tail = score_main


class LinearGaussianFullyAdapted(object):
    """The linear Gaussian model run as a fully adapted filter (csrc/pf_model.cuh, model id 2), operation for
    operation: proposal p(x_t | x_{t-1}, y_t), weight p(y_{t+1} | x_t).  flps_generic runs it on the observations
    shifted by one (obs[1:]); log_p_y1 adds the first observation's term.  No score terms (gradient rows 0)."""
    n_params = 3
    reference_indexing = False

    def __init__(self, params):
        self.phi, self.sv, self.se = [float(p) for p in params[:3]]
        s2 = self.sv * self.sv + self.se * self.se
        self.k = (self.sv * self.sv) / s2
        self.sdp = np.sqrt((self.sv * self.sv) * (self.se * self.se) / s2)
        self.inv_s2 = 1.0 / s2
        self.log_s = 0.5 * np.log(s2)

    def initial_state(self):
        return 0.0

    def propagate(self, xp, y_now, u):
        m = self.phi * xp
        return (m + self.k * (y_now - m)) + self.sdp * u

    def logw(self, x, y_next):
        r = y_next - self.phi * x
        return (-0.91893853320467267 - self.log_s) - (0.5 * (r * r)) * self.inv_s2

    def score_main(self, curr, nxt, y):
        return np.zeros((4,) + np.shape(curr))

    score_tail = score_main


def log_p_y1(obs, sv, se):
    """log p(y_1 | x_0 = 0) = log N(obs[1]; 0, sv^2 + se^2): the term the fully adapted filter's estimate of
    log p(y_2 .. y_T | y_1) lacks (x_0 = 0, so phi does not enter)."""
    s2 = sv * sv + se * se
    return -0.5 * np.log(2.0 * np.pi * s2) - 0.5 * float(obs[1]) ** 2 / s2


def systematic_corr(w, rnd):
    """:694-715 with Q3 (cum[0] is not normalised); the pointer walk = first index whose running maximum
    of the cumulative weights reaches the point."""
    n = w.shape[0]
    cum = np.cumsum(w)
    cum[1:] = cum[1:] / cum[-1]
    cp = (rnd + np.arange(n, dtype=np.float64)) / n
    return np.minimum(np.searchsorted(np.maximum.accumulate(cum), cp, side="left"), n - 1).astype(np.int32)


def flps_generic(model, obs, rvr, rvp, n_particles, lag=10, dumps=False):
    """Returns filt, smo, log_like, gradient [4][NOBS], traj (+ X, A, W when dumps).

    model.reference_indexing True (SV): the reference's pairing, quirks Q5 / Q6.  False (the linear Gaussian models):
    the pair (x_t, x_{t+1}), t = 0 .. NOBS-2, adds score(x_t, x_{t+1}, obs[t+1]) once, into gradient slot t+1 (slot 0
    stays 0), weighted by the generation at which it is read: W_{t+L-1} in the main loop, W_{NOBS-1} in the tail;
    smo[t] = E[x_t] under the same weights, every slot once (the tail starts one step after the last main-loop slot).
    """
    obs = np.asarray(obs, dtype=np.float64)
    nobs, n, L = obs.shape[0], int(n_particles), int(lag)
    ref = model.reference_indexing
    U = np.asarray(rvp, dtype=np.float64).reshape(n, nobs)        # rvp[i + j * NOBS]
    X = np.zeros((nobs, n))
    W = np.zeros((nobs, n))
    A = np.zeros((nobs, n), dtype=np.int32)
    filt, smo, traj = np.zeros(nobs), np.zeros(nobs), np.zeros(nobs)
    grad = np.zeros((4, nobs))
    x0 = model.initial_state()
    X[0] = x0
    W[0] = 1.0 / n
    A[0] = np.arange(n)
    ph = np.zeros((L, n))                                          # ph[k][j]: ancestor k steps back of sorted particle j
    ph[0] = x0
    filt[0] = np.sum(W[0] * X[0])
    traj[0] = x0
    log_like = 0.0
    for i in range(1, nobs):
        anc = systematic_corr(W[i - 1], rvr[i])
        xnew = model.propagate(X[i - 1][anc], obs[i - 1], U[:, i])
        order = np.argsort(xnew, kind="stable")
        X[i] = xnew[order]
        A[i] = anc[order]
        oph = ph.copy()
        ph[0] = X[i]
        ph[1:] = oph[:-1][:, A[i]]
        lw = model.logw(X[i], obs[i])
        mx = np.max(lw)                                            # (Q4: any shift cancels)
        sh = np.exp(lw - mx)
        nf = np.sum(sh)
        W[i] = sh / nf
        filt[i] = np.sum(W[i] * X[i])
        traj[i] = X[i][0]                                          # Q11
        if ref and i >= L:
            tt = i - L + 1
            curr, nxt = ph[L - 1], ph[L - 2]
            smo[tt] += np.sum(W[i] * curr)
            grad[:, tt] += np.sum(model.score_main(curr, nxt, obs[i - L]) * W[i], axis=1)   # Q5
        elif not ref and i >= L - 1:
            tt = i - L + 1                                         # pair (tt, tt + 1), tt = 0 included
            curr, nxt = ph[L - 1], ph[L - 2]
            smo[tt] += np.sum(W[i] * curr)
            grad[:, tt + 1] += np.sum(model.score_main(curr, nxt, obs[tt + 1]) * W[i], axis=1)
        log_like += mx + np.log(nf) - np.log(float(n))
    if ref:
        for i in range(nobs - L, nobs):                            # tail, :540-562 (Q6)
            idx = nobs - i - 1
            curr = ph[idx]
            smo[i] += np.sum(W[nobs - 1] * curr)
            if idx - 1 >= 0:
                nxt = ph[idx - 1]
                y1 = obs[i - 1] if i - 1 >= 0 else obs[i - 1 + nobs]
                if i - L + 1 >= 0:                                 # slot < 0 (nobs <= 2L - 2): dropped, not wrapped (DESIGN §2)
                    grad[:, i - L + 1] += np.sum(model.score_tail(curr, nxt, y1) * W[i], axis=1)
    else:
        for t in range(nobs - L + 1, nobs):                        # tail: final weights, one step after the main loop
            k = nobs - 1 - t
            smo[t] += np.sum(W[nobs - 1] * ph[k])
            if k >= 1:
                grad[:, t + 1] += np.sum(model.score_tail(ph[k], ph[k - 1], obs[t + 1]) * W[nobs - 1], axis=1)
    out = dict(filt=filt, smo=smo, log_like=float(log_like), gradient=grad, traj=traj)
    if dumps:
        out.update(X=X, A=A, W=W)
    return out


def kalman_loglike(obs, phi, sv, se):
    """Exact log-likelihood of obs[1:] for the linear Gaussian model started at x_0 = 0 (point mass), the
    convention of flps_generic: obs[0] is not weighted, obs[i] is the measurement of x_i."""
    m, p, ll = 0.0, 0.0, 0.0
    for y in np.asarray(obs, dtype=np.float64)[1:]:
        m, p = phi * m, phi * phi * p + sv * sv
        s = p + se * se
        ll += -0.5 * np.log(2.0 * np.pi * s) - 0.5 * (y - m) ** 2 / s
        k = p / s
        m, p = m + k * (y - m), (1.0 - k) * p
    return ll
