#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ from the REFERENCE ITSELF.

Run in the build container only (needs /root/reference and oracle/_ref built by
oracle/build_ref.py).  The reference ships no tests or fixtures (SURVEY.md section 4),
so parity is pinned by executing its own compiled Cython kernels and Python estimator
classes on seeded inputs and committing the outputs.  Inputs are NOT stored where
they can be regenerated bit-exactly from a NumPy ``RandomState`` seed
(``golden_inputs.py`` holds the generators shared with the tests).

Files written:
  sv_kernels.npz      flps_sv_corr / bpf_sv_corr outputs (stochastic_volatility.pyx:61,205)
  re_kernels.npz      importance_discrete outputs (random_effects.pyx:21)
  ss_kernels.npz      stratified indices (subsampling.pyx:34)
  estimators.npz      results dicts of ParticleMethodsCython / ImportanceSamplingCython /
                      DirectComputation driven through the reference's Python classes
                      (state/particle_methods/cython.py, state/importance_sampling/cython.py,
                      state/direct/standard.py, models/logistic_regression.py)
  qn_chain.npz        estimator calls recorded from a short run of the reference's unmodified
                      QuasiNewtonMetropolisHastings (parameter/mcmc/mh_quasi_newton.py)
"""
import os
import sys
import types
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, HERE)

import build_ref  # noqa: E402
import golden_inputs as gi  # noqa: E402

REF_PY = os.path.join(build_ref.REF_ROOT, "python")


# ------------------------------------------------------------------ kernels
def gen_sv_kernels():
    out = {}
    for (n, nobs, lag, seeds) in gi.SV_KERNEL_CASES:
        ref = build_ref.load("sv", n, nobs, lag)
        assert ref is not None, "build oracle/_ref first"
        assert tuple(ref.get_settings()) == (nobs, n, lag)
        for seed in seeds:
            obs, params, rvr, rvp = gi.sv_inputs(n, nobs, seed)
            tag = "n%d_t%d_l%d_s%d" % (n, nobs, lag, seed)
            for hess in (0, 1):
                r = ref.flps_sv_corr(obs, params, rvr, np.ascontiguousarray(rvp), hess)
                pre = "flps_%s_h%d_" % (tag, hess)
                out[pre + "filt"] = np.array(r[0], dtype=np.float64)
                out[pre + "smo"] = np.array(r[1], dtype=np.float64)
                out[pre + "log_like"] = np.float64(r[2])
                out[pre + "gradient"] = np.array(r[3], dtype=np.float64)
                out[pre + "traj"] = np.array(r[4], dtype=np.float64)
                out[pre + "hess1"] = np.array(r[5], dtype=np.float64)
                out[pre + "hess2"] = np.array(r[6], dtype=np.float64)
            if n <= 1024:
                r = ref.bpf_sv_corr(obs, params, rvr, np.ascontiguousarray(rvp))
                pre = "bpf_%s_" % tag
                out[pre + "filt"] = np.array(r[0], dtype=np.float64)
                out[pre + "log_like"] = np.float64(r[1])
                out[pre + "traj"] = np.array(r[2], dtype=np.float64)
            print("sv", tag, "ll", out["flps_%s_h0_log_like" % tag])
    np.savez_compressed(os.path.join(HERE, "sv_kernels.npz"), **out)


def gen_re_kernels():
    out = {}
    for (n, nobs, seeds) in gi.RE_KERNEL_CASES:
        ref = build_ref.load("re", n, nobs)
        assert tuple(ref.get_settings()) == (nobs, n)
        for seed in seeds:
            obs, params, rvr, rvp = gi.re_inputs(n, nobs, seed)
            r = ref.importance_discrete(obs, params, rvr, np.ascontiguousarray(rvp))
            pre = "is_n%d_t%d_s%d_" % (n, nobs, seed)
            out[pre + "filt"] = np.array(r[0], dtype=np.float64)
            out[pre + "log_like"] = np.float64(r[1])
            out[pre + "traj"] = np.array(r[2], dtype=np.float64)
            out[pre + "gradient"] = np.array(r[3], dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, "re_kernels.npz"), **out)


def gen_ss_kernels():
    out = {}
    for (m, n, seeds) in gi.SS_KERNEL_CASES:
        ref = build_ref.load("ss", m, n)
        assert tuple(ref.get_settings()) == (n, m)
        for seed in seeds:
            r = gi.ss_inputs(m, seed)
            out["strat_m%d_n%d_s%d" % (m, n, seed)] = np.array(ref.stratified(r), dtype=np.int32)
    np.savez_compressed(os.path.join(HERE, "ss_kernels.npz"), **out)


# ------------------------------------------------------- reference Python layer
def import_reference_python(sv=(75, 361, 10), re=(100, 100), ss=(5500, 110000)):
    """Import the reference's Python packages with the four shims of SURVEY.md section 8c
    (no edits to reference logic) and our size-variant builds of its Cython kernels."""
    np.float = float  # removed NumPy alias used at particle_methods/cython.py:49,79
    for name in ("quandl", "matplotlib", "matplotlib.pylab", "palettable",
                 "palettable.colorbrewer", "palettable.colorbrewer.qualitative"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["palettable.colorbrewer.qualitative"].Dark2_8 = types.SimpleNamespace(
        mpl_colors=[(0, 0, 0)] * 8)
    sys.modules["matplotlib"].pylab = sys.modules["matplotlib.pylab"]
    if REF_PY not in sys.path:
        sys.path.insert(0, REF_PY)
    warnings.filterwarnings("ignore", category=SyntaxWarning)
    import state  # noqa: F401
    import state.particle_methods  # noqa: F401
    import state.importance_sampling  # noqa: F401
    import state.direct  # noqa: F401
    sys.modules["state.particle_methods.stochastic_volatility"] = build_ref.load("sv", *sv)
    sys.modules["state.importance_sampling.random_effects"] = build_ref.load("re", *re)
    sys.modules["state.direct.subsampling"] = build_ref.load("ss", *ss)
    import state.base_state_inference  # noqa: F401  (arms warnings->errors)
    warnings.filterwarnings("ignore", category=SyntaxWarning)
    warnings.filterwarnings("ignore", category=DeprecationWarning)


def make_ref_sv_model(nobs, params):
    from models.stochastic_volatility import StochasticVolatilityModel
    model = StochasticVolatilityModel()
    y = gi.sv_obs(nobs)
    model.obs = np.array(y, copy=True).reshape((nobs, 1))
    model.no_obs = nobs - 1
    for k, v in zip(("mu", "phi", "sigma_v", "rho"), params):
        model.params[k] = float(v)
    model.fix_true_params()
    model.create_inference_model(params_to_estimate=("mu", "phi", "sigma_v", "rho"))
    return model


def _prior_terms(model, out, pre):
    pg = model.log_prior_gradient()
    ph = model.log_prior_hessian()
    if isinstance(pg, dict):
        out[pre + "prior_grad"] = np.array([pg[k] for k in model.params.keys()], dtype=np.float64)
        out[pre + "prior_hess"] = np.array([ph[k] for k in model.params.keys()], dtype=np.float64)
    else:
        out[pre + "prior_grad"] = np.array(pg, dtype=np.float64)
        out[pre + "prior_hess"] = np.array(ph, dtype=np.float64)


def gen_estimators():
    import_reference_python()
    from state.particle_methods.cython import ParticleMethodsCython
    from state.importance_sampling.cython import ImportanceSamplingCython
    from state.direct.standard import DirectComputation
    from models.random_effects import RandomEffectsModel
    from models.logistic_regression import LogisticRegressionModel
    out = {}

    # --- SV particle smoother / filter through ParticleMethodsCython
    n, nobs, lag = 75, 361, 10
    for ci, params in enumerate(gi.SV_ESTIMATOR_PARAMS):
        model = make_ref_sv_model(nobs, params)
        est = ParticleMethodsCython(model)
        assert est.dim_rvs == (nobs, n + 1)
        for hess in (0, 1):
            model.using_gradients = True
            model.using_hessians = bool(hess)
            rvs = gi.sv_rvs(n, nobs, seed=1000 + ci)
            ok = est.smoother(model, rvs={"rvs": rvs})
            pre = "sv_smoother_c%d_h%d_" % (ci, hess)
            out[pre + "ok"] = np.bool_(ok)
            for k in ("filt_state_est", "state_trajectory", "smo_state_est", "log_like",
                      "gradient_internal", "log_joint_gradient_estimate"):
                out[pre + k] = np.array(est.results[k], dtype=np.float64)
            if hess:
                for k in ("log_joint_hessian_estimate", "hessian_internal",
                          "hessian_internal_noprior"):
                    out[pre + k] = np.array(est.results[k], dtype=np.float64)
            _prior_terms(model, out, pre)
            est.results = {}
        ok = est.filter(model, rvs={"rvs": gi.sv_rvs(n, nobs, seed=1000 + ci)})
        pre = "sv_filter_c%d_" % ci
        out[pre + "ok"] = np.bool_(ok)
        for k in ("filt_state_est", "state_trajectory", "log_like"):
            out[pre + k] = np.array(est.results[k], dtype=np.float64)

    # --- random effects through ImportanceSamplingCython
    n, nobs = 100, 100
    for ci, params in enumerate(gi.RE_ESTIMATOR_PARAMS):
        model = RandomEffectsModel()
        model.params["mu"] = float(params[0])
        model.params["sigma"] = float(params[1])
        model.obs = gi.re_obs(nobs)
        model.no_obs = nobs
        model.fix_true_params()
        model.create_inference_model()
        model.using_gradients = True
        model.using_hessians = False
        est = ImportanceSamplingCython(model)
        rvs = gi.re_rvs(n, nobs, seed=2000 + ci)
        ok = est.smoother(model, rvs={"rvs": rvs})
        pre = "re_smoother_c%d_" % ci
        out[pre + "ok"] = np.bool_(ok)
        for k in ("filt_state_est", "state_trajectory", "log_like", "gradient_internal",
                  "log_joint_gradient_estimate"):
            out[pre + k] = np.array(est.results[k], dtype=np.float64)
        _prior_terms(model, out, pre)

    # --- logistic regression through DirectComputation (shipped sizes 110000 / 5500)
    n_data, d, m = 110000, gi.LOGIT_D, 5500
    x, y, beta = gi.logit_data(n_data, d)
    model = LogisticRegressionModel(no_regressors=d)
    model.load_data_object({"x": x, "y": y})
    model.params = np.array(beta, copy=True)
    model.params_prior = gi.logit_prior(d)
    model.true_params = np.array(beta, copy=True)
    model.create_inference_model()   # as scripts/helper_higgs.py:50 does
    model.using_gradients = True
    est = DirectComputation(model)
    assert est.dim_rvs == m
    for ci in range(2):
        u = gi.logit_u(m, seed=3000 + ci)
        for hess in (False, True):
            ok = est.smoother(model, compute_hessian=hess, rvs={"rvs": u})
            pre = "logit_smoother_c%d_h%d_" % (ci, int(hess))
            out[pre + "ok"] = np.bool_(ok)
            out[pre + "log_like"] = np.float64(est.results["log_like"])
            out[pre + "gradient"] = np.array(est.results["gradient"], dtype=np.float64)
            out[pre + "gradient_internal"] = np.array(est.results["gradient_internal"],
                                                      dtype=np.float64)
            if hess:
                out[pre + "hessian"] = np.array(est.results["hessian"], dtype=np.float64)
                out[pre + "hessian_internal"] = np.array(est.results["hessian_internal"],
                                                         dtype=np.float64)
            out[pre + "prior_grad"] = np.array(model.log_prior_gradient(), dtype=np.float64)
            out[pre + "prior_hess"] = np.array(model.log_prior_hessian(), dtype=np.float64)
        ok = est.filter(model, rvs={"rvs": u})
        out["logit_filter_c%d_log_like" % ci] = np.float64(est.results["log_like"])
    np.savez_compressed(os.path.join(HERE, "estimators.npz"), **out)
    print("estimators: %d arrays" % len(out))


def gen_qn_chain(no_iters=16):
    """Run the reference's QuasiNewtonMetropolisHastings UNMODIFIED on the SV model
    (T=360, N=75) and record what it asked of the estimator."""
    import_reference_python()
    from state.particle_methods.cython import ParticleMethodsCython
    from parameter.mcmc.mh_quasi_newton import QuasiNewtonMetropolisHastings
    n, nobs = 75, 361
    np.random.seed(87655678)
    model = make_ref_sv_model(nobs, (0.2, 0.9, 0.4, -0.5))
    est = ParticleMethodsCython(model)
    calls = []
    orig = est.smoother

    def recording_smoother(mdl, **kw):
        ok = orig(mdl, **kw)
        calls.append(dict(params=np.array(mdl.get_all_params(), dtype=np.float64),
                          rvs=np.array(kw["rvs"]["rvs"], dtype=np.float64),
                          ok=bool(ok),
                          log_like=float(est.results.get("log_like", np.nan)),
                          gradient_internal=np.array(est.results.get("gradient_internal",
                                                                     np.full(4, np.nan)),
                                                     dtype=np.float64)))
        return ok

    est.smoother = recording_smoother
    hessian_guess = np.diag((0.01, 0.01, 0.01, 0.001))
    settings = {"no_iters": no_iters, "no_burnin_iters": 8, "adapt_step_size": True,
                "adapt_step_size_initial": 0.1, "adapt_step_size_rate": 0.5,
                "adapt_step_size_target": 0.2, "initial_params": (2.0, 0.9, 0.4, -0.2),
                "no_iters_between_progress_reports": 1000, "correlated_rvs": True,
                "correlated_rvs_sigma": 0.5, "memory_length": 5,
                "accept_first_iterations": 5, "hessian": hessian_guess,
                "hess_corr_fallback": hessian_guess, "hess_corr_method": "flip"}
    sampler = QuasiNewtonMetropolisHastings(model, settings, qn_method="bfgs")
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        try:
            sampler.run(est)
        except Exception as exc:  # post-run statistics may choke on so short a chain
            if len(calls) < 2 * no_iters:
                raise
            sys.stderr.write("qn_chain: run() raised after the last iteration: %r\n" % (exc,))
    out = {"n_calls": np.int64(len(calls))}
    keep_rvs = 4     # 211 KB compressed each (random fp64 barely compresses); keeps the file under 1 MB
    for k, c in enumerate(calls):
        out["call%d_params" % k] = c["params"]
        out["call%d_ok" % k] = np.bool_(c["ok"])
        out["call%d_log_like" % k] = np.float64(c["log_like"])
        out["call%d_gradient_internal" % k] = c["gradient_internal"]
        if k < keep_rvs:
            out["call%d_rvs" % k] = c["rvs"]
    np.savez_compressed(os.path.join(HERE, "qn_chain.npz"), **out)
    print("qn_chain: %d estimator calls recorded" % len(calls))


if __name__ == "__main__":
    which = sys.argv[1:] or ["sv", "re", "ss", "est", "qn"]
    if "sv" in which:
        gen_sv_kernels()
    if "re" in which:
        gen_re_kernels()
    if "ss" in which:
        gen_ss_kernels()
    if "est" in which:
        gen_estimators()
    if "qn" in which:
        gen_qn_chain()
