"""The two CPU restatements of the SV smoother over every lag and every short series the entries accept.

pmmh_flps_sv_corr takes 2 <= lag <= 63 and n_obs >= lag + 1.  For n_obs <= 2 lag - 2 the reference's tail
(stochastic_volatility.pyx:540-562, quirk Q6) indexes gradient slot i - LAG + 1 < 0 for its first steps: undefined in
the reference, whose buffers are C arrays.  The rule every restatement and every kernel follows (DESIGN.md section 2):
those gradient terms are dropped; the Hessian sums, which have no slot, keep them.

- guard: oracle_flps_sv_corr writes nothing outside its outputs (canaries before and after every buffer), with and
  without the Hessian, down to N = 1;
- agreement: the C oracle and oracle/generic_pf.py (SvLeverage) give the same ancestors and estimates, and the same
  gradient slots stay exactly zero (the visible effect of the rule);
- mutation: a tail that wraps the slot (slot n_obs + tt, what NumPy's negative index would do) or writes it into slot 0
  fails the agreement check.
"""
import ctypes

import numpy as np
import pytest

import golden_inputs as gi

LAGS = (2, 3, 4, 9, 10, 11, 13, 14, 31, 32, 33, 62, 63)
NS = (1, 5, 37, 300)
PAD = 64
CANARY = 0.5 ** 20         # small: a stray += of any term changes it
ICANARY = -123456789


def _nobs_list(lag):
    return sorted({m for m in (lag + 1, lag + 2, 2 * lag - 2, 2 * lag - 1, 2 * lag, 2 * lag + 1) if m >= lag + 1})


SHAPES = [(lag, m) for lag in LAGS for m in _nobs_list(lag)]


def _inputs(lag, nobs, n):
    return gi.sv_inputs(n, nobs, lag + nobs)


def _padded(size, dtype=np.float64):
    buf = np.full(size + 2 * PAD, ICANARY if dtype == np.int32 else CANARY, dtype=dtype)
    return buf, buf[PAD:PAD + size]


@pytest.mark.parametrize("lag,nobs", SHAPES, ids=["L%d-T%d" % s for s in SHAPES])
def test_oracle_writes_only_its_outputs(lag, nobs):
    """every output buffer (and the X / A / W dumps) framed by PAD canaries on each side: all intact after the call"""
    import oracle
    lib = oracle.lib()
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)
    for n in NS:
        obs, params, rvr, rvp = _inputs(lag, nobs, n)
        for hess in (0, 1):
            sizes = dict(filt=nobs, smo=nobs, ll=1, grad=4 * nobs, traj=nobs, h1=16, h2=16, X=nobs * n, W=nobs * n)
            bufs = {k: _padded(s) for k, s in sizes.items()}
            bufs["A"] = _padded(nobs * n, np.int32)
            bufs["info"] = _padded(4, np.int32)
            ptr = {k: v[1].ctypes.data_as(ip if v[1].dtype == np.int32 else dp) for k, v in bufs.items()}
            rc = lib.oracle_flps_sv_corr(
                obs.ctypes.data_as(dp), params.ctypes.data_as(dp), rvr.ctypes.data_as(dp), rvp.ctypes.data_as(dp),
                ctypes.c_int(n), ctypes.c_int(nobs), ctypes.c_int(lag), ctypes.c_int(hess), ptr["filt"], ptr["smo"],
                ptr["ll"], ptr["grad"], ptr["traj"], ptr["h1"], ptr["h2"], ptr["X"], ptr["A"], ptr["W"], ptr["info"])
            assert rc == 0
            for k, (full, _) in bufs.items():
                c = ICANARY if full.dtype == np.int32 else CANARY
                for side, pad in (("before", full[:PAD]), ("after", full[-PAD:])):
                    assert np.all(pad == c), "oracle wrote %s %s (lag %d, n_obs %d, N %d, hess %d)" % (
                        side, k, lag, nobs, n, hess)
            out = bufs["grad"][1]
            assert np.all(np.isfinite(out))
            if hess:
                assert np.all(np.isfinite(bufs["h1"][1])) and np.all(np.isfinite(bufs["h2"][1]))


def disagreement(ref, got):
    """what differs between two runs of the smoother (empty: they agree): ancestors exact, X and every estimate
    within 1e-12 of its largest entry, the same exactly-zero gradient slots"""
    bad = []
    if not np.array_equal(got["A"][1:], ref["A"][1:]):
        bad.append("ancestors")
    for k in ("X", "filt", "smo", "traj", "gradient"):
        scale = max(float(np.max(np.abs(ref[k]))), 1e-300)
        if not np.max(np.abs(got[k] - ref[k])) <= 1e-12 * scale:
            bad.append(k)
    if not abs(got["log_like"] - ref["log_like"]) <= 1e-12 * abs(ref["log_like"]):
        bad.append("log_like")
    if not np.array_equal(got["gradient"] == 0.0, ref["gradient"] == 0.0):
        bad.append("zero slots")
    return bad


def _runs(lag, nobs, n):
    import generic_pf as gp
    import oracle
    obs, params, rvr, rvp = _inputs(lag, nobs, n)
    ref = oracle.flps_sv_corr(obs, params, rvr, rvp, n, lag, 0, dumps=True)
    got = gp.flps_generic(gp.SvLeverage(params), obs, rvr, rvp, n, lag, dumps=True)
    return (obs, params), ref, got


def tail_terms(model, obs, X, A, W, lag):
    """{tt: gradient term} of the reference's tail steps (slot tt = i - lag + 1, negative where the rule drops the
    term), restated from a run's history: the lineage of the final generation, weighted by W_i (quirk Q6)"""
    nobs, n = X.shape
    ph = np.zeros((lag, n))
    idx = np.arange(n)
    for k in range(lag):
        ph[k] = X[nobs - 1 - k][idx]
        idx = A[nobs - 1 - k][idx]
    out = {}
    for i in range(nobs - lag, nobs):
        k = nobs - i - 1
        if k >= 1:
            out[i - lag + 1] = np.sum(model.score_tail(ph[k], ph[k - 1], obs[i - 1]) * W[i], axis=1)
    return out


def dropped_terms(model, obs, X, A, W, lag):
    return {tt: v for tt, v in tail_terms(model, obs, X, A, W, lag).items() if tt < 0}


@pytest.mark.parametrize("lag,nobs", SHAPES, ids=["L%d-T%d" % s for s in SHAPES])
def test_restatements_agree(lag, nobs):
    """the C oracle and the NumPy restatement agree at every N, zero slots included.  Those are the last lag - 1
    slots (no pair is read there), and slot 0 from n_obs = 2 lag on (the tail's first slot is n_obs - 2 lag + 1)"""
    zero = set(range(nobs - lag + 1, nobs)) | ({0} if nobs >= 2 * lag else set())
    for n in NS:
        _, ref, got = _runs(lag, nobs, n)
        assert disagreement(ref, got) == [], (lag, nobs, n, disagreement(ref, got))
        assert set(np.nonzero(np.all(ref["gradient"] == 0.0, axis=0))[0]) == zero


MUTATION_SHAPES = [s for s in SHAPES if s[1] <= 2 * s[0] - 2]


@pytest.mark.parametrize("lag,nobs", MUTATION_SHAPES, ids=["L%d-T%d" % s for s in MUTATION_SHAPES])
def test_a_tail_that_keeps_the_dropped_terms_fails(lag, nobs):
    """adding the dropped terms back, wrapped to slot n_obs + tt or into slot 0, is caught by the agreement check"""
    import generic_pf as gp
    for n in (5, 37):
        (obs, params), ref, got = _runs(lag, nobs, n)
        terms = dropped_terms(gp.SvLeverage(params), obs, got["X"], got["A"], got["W"], lag)
        assert sorted(terms) == list(range(nobs - 2 * lag + 1, 0))
        assert all(np.max(np.abs(v)) > 0.0 for v in terms.values())
        for where in ("wrap", "slot0"):
            mutated = dict(got, gradient=got["gradient"].copy())
            for tt, v in terms.items():
                mutated["gradient"][:, nobs + tt if where == "wrap" else 0] += v
            assert disagreement(ref, mutated) != [], (where, lag, nobs, n)


def test_tail_terms_restate_the_tail():
    """the helper reproduces the restatements' tail: at n_obs = 2 lag - 1 slot 0 holds the tail's term tt = 0 alone,
    and no term is dropped; at n_obs = lag + 1 the terms tt = 2 - lag .. -1 are"""
    import generic_pf as gp
    lag, n = 10, 37
    (obs, params), ref, got = _runs(lag, 2 * lag - 1, n)
    terms = tail_terms(gp.SvLeverage(params), obs, got["X"], got["A"], got["W"], lag)
    assert sorted(terms) == list(range(0, lag - 1))
    assert np.max(np.abs(terms[0] - ref["gradient"][:, 0])) <= 1e-12 * np.max(np.abs(ref["gradient"]))
    assert np.max(np.abs(terms[0])) > 0.0
    (obs, params), _, got = _runs(lag, lag + 1, n)
    assert sorted(dropped_terms(gp.SvLeverage(params), obs, got["X"], got["A"], got["W"], lag)) == list(
        range(2 - lag, 0))
