"""Auxiliary variables u that drive the particle sort of the smoother kernels into its edges.

Every kernel replaces the reference's qsort of the children's values (stochastic_volatility.pyx:23-52) with a
sort that bins the values over a predicted range and ranks inside a bin.  These builders make the inputs that
reach each part of such a sort on purpose; each returns ``(u, rvp)``: u in the device's time-major layout
[n_obs][N] and the reference's flat rvp[t + j * n_obs] (the same numbers).  Row 0 is never read (the initial
generation is one point, quirk Q1); row t >= 1 drives the propagation into generation t (pmmh_oracle.c:319,
generic_pf.py's U[:, i]).

- ``sibling_ties``: on every second step from generation 2 on, runs of m consecutive children share one u.
  Children are numbered by systematic resampling, so the children of one parent are consecutive, and siblings
  with one u have equal values.  The steps in between are tie-free, so the parents of a tied step are distinct
  values: every exact tie is between children of one parent, whose order no output can tell.
- ``tie_group``: g children of generation 1 get u = +5 exactly, every other u of that row is N(0, 1) truncated to
  |u| < 4.  Generation 0 is one point, so the group is g equal values alone in its bin, whatever the kernel's
  bin width (at most 1 predicted sd); its members come from different (equal-valued) parents.
- ``outliers``: per step, six children at u = -40, -12, -7, +7, +12, +40; the first child (whose parent is the
  smallest particle) takes -40 and the last (the largest parent) +40, so those two land at sorted positions 0 and
  N - 1.  All of them fall outside a predicted range of +-6.5 sd.
- ``near_ties``: runs of m consecutive children get u0 + k delta, k = 0 .. m-1, with delta * sd = ``ulps`` units in
  the last place of ``xscale``: siblings differ by a few ulp but never tie.
- ``plain``: N(0, 1); with a small sigma_v (the caller's parameters) it makes the narrow cloud.
"""
import numpy as np

PATTERNS = ("plain", "sibling_ties", "tie_group", "outliers", "near_ties")
GROUP_U = 5.0                 # the tie group's u: inside +-6.5 sd, and 1 sd clear of every other u of its row
TRUNC = 4.0                   # |u| bound of the rest of the group's row
OUTLIER_U = (-40.0, -12.0, -7.0, 7.0, 12.0, 40.0)


def flat_rvp(u):
    """time-major u[t][j] -> the reference's flat rvp[t + j * n_obs]"""
    return np.ascontiguousarray(np.asarray(u, dtype=np.float64).T).reshape(-1)


def _truncated_normal(rs, size, bound):
    z = rs.standard_normal(size)
    bad = np.abs(z) >= bound
    while bad.any():
        z[bad] = rs.standard_normal(int(bad.sum()))
        bad = np.abs(z) >= bound
    return z


def build(pattern, n, n_obs, seed, m=2, g=2, ulps=2, sd=1.0, xscale=1.0):
    """(u [n_obs][n], rvp [n_obs * n]) of one pattern (see the module docstring).  m: run length (sibling_ties,
    near_ties); g: tie group size (tie_group); sd / xscale: the propagation sd and a bound on |x| (near_ties)."""
    rs = np.random.RandomState(seed)
    u = rs.standard_normal((n_obs, n))
    if pattern == "plain":
        pass
    elif pattern == "sibling_ties":
        assert m >= 2
        for t in range(2, n_obs, 2):
            u[t] = np.repeat(u[t, ::m], m)[:n]
    elif pattern == "tie_group":
        assert 2 <= g < n and n_obs >= 2
        u[1] = _truncated_normal(rs, n, TRUNC)
        u[1, rs.choice(n, g, replace=False)] = GROUP_U
    elif pattern == "outliers":
        assert n > 2 * len(OUTLIER_U)
        for t in range(1, n_obs):
            inner = 1 + rs.choice(n - 2, len(OUTLIER_U) - 2, replace=False)
            u[t, 0], u[t, n - 1] = OUTLIER_U[0], OUTLIER_U[-1]
            u[t, inner] = OUTLIER_U[1:-1]
    elif pattern == "near_ties":
        assert m >= 2
        delta = ulps * np.spacing(float(xscale)) / sd
        k = np.arange(n) % m
        for t in range(1, n_obs):
            u[t] = np.repeat(u[t, ::m], m)[:n] + k * delta
    else:
        raise ValueError("unknown pattern %r" % (pattern,))
    u = np.ascontiguousarray(u)
    return u, flat_rvp(u)


def sv_child_sd(params):
    """the SV propagation sd sqrt(1 - rho^2) sigma_v (pmmh_oracle.c:318)"""
    return float(np.sqrt(1.0 - params[3] ** 2) * params[2])


def sv_xscale(params):
    """a bound on |x| of the SV cloud: |mu| + 8 stationary sd"""
    mu, phi, sv = params[:3]
    return float(abs(mu) + 8.0 * sv / np.sqrt(1.0 - phi * phi))
