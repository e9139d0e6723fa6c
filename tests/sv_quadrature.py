"""TEST INFRASTRUCTURE ONLY -- exact (fine-grid quadrature) fixed-lag targets for a scalar-state model, the non-Gaussian
counterpart of oracle/kalman.py.  Nothing under pmmh-qn_b200/ imports it.

Model (the kernels' convention): x_0 = model.initial_state() (a point mass), x_t | x_{t-1} ~ N(m(x_{t-1}, obs[t-1]),
sd^2) with m = model.propagate(x, y, 0), y_t = obs[t] weighted by exp(model.logw(x_t, y_t)) for t >= 1; obs[0] is not
weighted.  The densities are tabulated on a uniform grid and integrated with the trapezoid rule on a range that holds
all the mass, which converges geometrically for these smooth, fast-decaying integrands: with the linear Gaussian
callbacks the results match oracle/kalman.py to within 1e-13 relative on the test series (log-likelihood 3e-14, filtered and
smoothed means and score slots 1e-15; tests/test_sv_exact_reference.py asserts 1e-11).

quadrature_targets returns
  * log_like = sum_{t >= 1} log p(y_t | y_1 .. y_t-1) (and x_0, obs[0]);
  * filt[t] = E[x_t | y_1 .. y_t];
  * per pair (x_t, x_t+1), t = 0 .. T-2, conditioned on exactly the observations its weights see,
    y_1 .. y_c(t), c(t) = min(t + lag - 1, T - 1): smo[t] = E[x_t | .], score[:, t] = E[s_t | .] and hess1[t] = E[H_t | .],
    where s_t / H_t are the model's pair hooks (score_main / hess_main with y = obs[t + pair_y], the first-pair hooks
    score_first / hess_first for t = 0 where the model has them), and with `hessian` hess1[t] = E[H_t | .] and
    hess2[t] = E[s_t s_t' + a_t s_t' + s_t a_t' | .], a_t(x_t) = E[s_0 + .. + s_t-1 | x_t, y_1 .. y_t] (the alpha of
    Louis' identity: the past is independent of later observations given x_t), computed by a forward recursion over
    the backward kernels p(x_t-1 | x_t, y_1 .. y_t-1);
and fd_gradient / fd_hessian differentiate log_like numerically over any parametrisation.
"""
import numpy as np


def _grid(lo, hi, m):
    x = np.linspace(lo, hi, m)
    w = np.full(m, x[1] - x[0])
    w[0] = w[-1] = 0.5 * (x[1] - x[0])
    return x, w


def _kernel(model, sd, xs, y_prev):
    """K[j, i] = N(x_j; m(x_i, y_prev), sd^2)"""
    m = model.propagate(xs, y_prev, 0.0)
    return np.exp(-0.5 * ((xs[:, None] - m[None, :]) / sd) ** 2) / (np.sqrt(2.0 * np.pi) * sd)


def _obs_density(model, xs, y):
    return np.exp(model.logw(xs, y))


def forward(model, sd, obs, xs, wq):
    """filtered densities f[t] on the grid (t >= 1; f[0] unused), predictive constants and log-likelihood"""
    obs = np.asarray(obs, dtype=np.float64)
    T = obs.shape[0]
    x0 = model.initial_state()
    f = np.zeros((T, xs.shape[0]))
    ll = 0.0
    for t in range(1, T):
        if t == 1:
            m = model.propagate(np.array([x0]), obs[0], 0.0)[0]
            pred = np.exp(-0.5 * ((xs - m) / sd) ** 2) / (np.sqrt(2.0 * np.pi) * sd)
        else:
            pred = _kernel(model, sd, xs, obs[t - 1]) @ (f[t - 1] * wq)
        un = pred * _obs_density(model, xs, obs[t])
        z = np.sum(un * wq)
        ll += np.log(z)
        f[t] = un / z
    return f, ll


def log_likelihood(model, sd, obs, xs, wq):
    return forward(model, sd, obs, xs, wq)[1]


def _pair_hook(model, name, t, curr, nxt, y):
    if t == 0 and hasattr(model, name + "_first"):
        return getattr(model, name + "_first")(nxt, y)
    return getattr(model, name + "_main")(curr, nxt, y)


def quadrature_targets(model, sd, obs, lag, lo, hi, m=801, pair_y=0, hessian=False):
    """module docstring; pair_y = 0: the pair (x_t, x_t+1) reads obs[t] (predictive pairing, the SV model), 1: obs[t+1]
    (exact pairing, the linear Gaussian bootstrap filter)"""
    obs = np.asarray(obs, dtype=np.float64)
    T, L = obs.shape[0], int(lag)
    xs, wq = _grid(lo, hi, m)
    f, ll = forward(model, sd, obs, xs, wq)
    x0 = model.initial_state()
    g = np.array([_obs_density(model, xs, obs[t]) if t >= 1 else np.ones_like(xs) for t in range(T)])
    filt = np.array([x0] + [np.sum(xs * f[t] * wq) for t in range(1, T)])
    smo, score = np.zeros(T), np.zeros((4, T))
    hess1, hess2 = np.zeros((T, 4, 4)), np.zeros((T, 4, 4))
    a = np.zeros((4, xs.shape[0]))                 # a_t on the grid (a_0 = 0)
    kernels = {}
    for t in range(T - 1):
        c = min(t + L - 1, T - 1)
        beta = np.ones_like(xs)                    # p(y_t+2 .. y_c | x_t+1) up to a constant
        for s in range(c, t + 1, -1):
            if s not in kernels:
                kernels[s] = _kernel(model, sd, xs, obs[s - 1])
            beta = kernels[s].T @ (g[s] * beta * wq)
            beta = beta / np.max(beta)
        y = obs[t + pair_y]
        if t == 0:
            # x_0 = x0: the joint is a density of x_1 alone
            m0 = model.propagate(np.array([x0]), obs[0], 0.0)[0]
            p1 = np.exp(-0.5 * ((xs - m0) / sd) ** 2) * g[1] * beta * wq
            p1 = p1 / np.sum(p1)
            smo[0] = x0
            curr, nxt, w = np.full_like(xs, x0), xs, p1
        else:
            if t + 1 not in kernels:
                kernels[t + 1] = _kernel(model, sd, xs, obs[t])
            joint = kernels[t + 1] * (f[t] * wq)[None, :] * (g[t + 1] * beta * wq)[:, None]   # [x_t+1, x_t]
            joint = joint / np.sum(joint)
            smo[t] = np.sum(joint.sum(axis=0) * xs)
            curr = np.broadcast_to(xs[None, :], joint.shape).ravel()
            nxt = np.broadcast_to(xs[:, None], joint.shape).ravel()
            w = joint.ravel()
        sc = _pair_hook(model, "score", t, curr, nxt, y)
        score[:, t] = np.sum(sc * w, axis=1)
        if hessian:
            hess1[t] = np.sum(_pair_hook(model, "hess", t, curr, nxt, y) * w, axis=2)
            al = np.zeros_like(sc) if t == 0 else np.broadcast_to(a[:, None, :], (4,) + joint.shape).reshape(4, -1)
            hess2[t] = np.einsum("an,bn,n->ab", sc, sc, w) + np.einsum("an,bn,n->ab", al, sc, w) + \
                np.einsum("an,bn,n->ab", sc, al, w)
            # a_t+1(x') = E[a_t(x_t) + s_t(x_t, x') | x_t+1 = x', y_1 .. y_t] (backward kernel: f_t(x) p(x' | x))
            if t == 0:
                a = sc.copy()
            else:
                bk = kernels[t + 1] * (f[t] * wq)[None, :]
                bk = bk / np.sum(bk, axis=1, keepdims=True)
                a = np.einsum("ji,aji->aj", bk, a[:, None, :] + sc.reshape((4,) + joint.shape))
    # the last state: smo[T - 1] = E[x_T-1 | y_1 .. y_T-1]
    smo[T - 1] = np.sum(xs * f[T - 1] * wq)
    out = dict(log_like=ll, filt=filt, smo=smo, score=score)
    if hessian:
        out["hess1"], out["hess2"] = hess1, hess2
    return out


def fd_gradient(make, theta, obs, lo, hi, m=801, h=1e-5):
    """central differences of log_like over theta; make(theta) -> (model, sd)"""
    theta = np.asarray(theta, dtype=np.float64)
    xs, wq = _grid(lo, hi, m)
    f = lambda p: log_likelihood(*make(p), obs, xs, wq)
    e = np.eye(theta.shape[0]) * h
    return np.array([(f(theta + e[a]) - f(theta - e[a])) / (2.0 * h) for a in range(theta.shape[0])])


def fd_hessian(make, theta, obs, lo, hi, m=801, h=1e-3):
    """central differences of log_like over theta (symmetrised)"""
    theta = np.asarray(theta, dtype=np.float64)
    xs, wq = _grid(lo, hi, m)
    f = lambda p: log_likelihood(*make(p), obs, xs, wq)
    d = theta.shape[0]
    e = np.eye(d) * h
    out = np.zeros((d, d))
    for a in range(d):
        for b in range(d):
            out[a, b] = (f(theta + e[a] + e[b]) - f(theta + e[a] - e[b]) - f(theta - e[a] + e[b])
                         + f(theta - e[a] - e[b])) / (4.0 * h * h)
    return 0.5 * (out + out.T)
