#!/usr/bin/env python
"""bench.py -- headline benchmark of the likelihood-estimation hot path (BASELINE.json).

Workload (config 2 of BASELINE.json, the size its target is quoted on): stochastic-volatility
fixed-lag particle smoother, T = 1000 returns, N = 2^20 particles, log-likelihood + gradient
(hess = 0), synthetic returns and u.  One "step" = one evaluation.  With --gpus N every rank
evaluates its own independent (theta, u) problem (chain-batched sharding, no collective on the
data path) => weak scaling; `value` is the whole-job particle-timesteps/s.

  python bench.py                      # 1 GPU, defaults
  torchrun ... bench.py --gpus N ...   # one rank per GPU (the driver launches this)
  python bench.py --impl reference     # the reference's own CPU implementation (oracle/_ref)
  python bench.py --dump-outputs DIR   # also write the estimates of the last timed step to DIR/*.npy

Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests", "golden")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

T_STEPS = 1000
NOBS = T_STEPS + 1
LAG = 10
PARAMS = (0.2, 0.9, 0.4, -0.5)
BYTES_PER_PARTICLE_STEP = 96          # SURVEY 8(d): 7s + 40 at s = 8 (filter + fixed-lag gradient)
KERNEL_NAMES = {1: "sv_pf_kernel<false> (general kernel)", 2: "sv_fast_kernel (exchange kernel)",
                3: "sv_chain_kernel", 4: "streaming kernels with path storage (sv_split.cu: children, "
                                         "lineage, fine histogram, offsets, scatter, rank, weights, finalize per time step)",
                5: "sv_grid_kernel (grid kernel: one persistent cooperative launch, one tile of the sorted "
                   "generation per SM, four grid barriers per time step)"}
METRIC = "particle_timesteps_per_sec"
UNIT = "particle-timesteps/s"


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------- clocks
class ClockSampler(object):
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, smax, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in out.splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8 or parts[0] != str(self.gpu_index):
                continue
            try:
                sm.append(float(parts[1]))
                smax = float(parts[2])
            except ValueError:
                continue
            for name, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- reference arm
def _ref_worker(args):
    """One evaluation of the reference's compiled flps_sv_corr (N=1024, T=1000) in this process."""
    seed, reps = args
    import build_ref
    import golden_inputs as gi
    ref = build_ref.load("sv", 1024, NOBS, LAG)
    obs = gi.sv_obs(NOBS)
    rvr, rvp = gi.split_particle(gi.sv_rvs(1024, NOBS, seed), NOBS)
    params = np.array(PARAMS)
    t0 = time.perf_counter()
    ll = 0.0
    for _ in range(reps):
        ll = ref.flps_sv_corr(obs, params, rvr, rvp, 0)[2]
    return time.perf_counter() - t0, float(ll)


def _port_worker(args):
    seed, n = args
    import golden_inputs as gi
    import oracle
    obs = gi.sv_obs(NOBS)
    rvr, rvp = gi.split_particle(gi.sv_rvs(n, NOBS, seed), NOBS)
    t0 = time.perf_counter()
    out = oracle.flps_sv_corr(obs, np.array(PARAMS), rvr, rvp, n, LAG, 0)
    return time.perf_counter() - t0, out["log_like"]


def _port_sample_worker(args):
    """The O(T N) oracle port at the headline N for a short series (same-config CPU number)."""
    seed, n, tsteps = args
    import oracle
    import golden_inputs as gi
    nobs = tsteps + 1
    rng = np.random.default_rng(seed)
    obs = gi.sv_obs(nobs)
    rvr = rng.random(nobs)
    rvp = rng.standard_normal(n * nobs)
    t0 = time.perf_counter()
    out = oracle.flps_sv_corr(obs, np.array(PARAMS), rvr, rvp, n, LAG, 0)
    return time.perf_counter() - t0, out["log_like"]


def cpu_port_same_config(n, tsteps=24):
    """All host cores, one independent N-particle evaluation per core over `tsteps` time steps."""
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cores = min(cores, 32)            # 92 MB of u per worker at N = 2^20; bounded fan-out
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_port_sample_worker, [(77 + w, n, tsteps) for w in range(cores)])
    wall = time.perf_counter() - t0
    inner = max(r[0] for r in res)
    return {"value": cores * n * tsteps / inner, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "oracle port (O(T N) restatement, oracle/pmmh_oracle.c) flps_sv_corr hess=0, N=%d, first %d time "
                      "steps, one independent evaluation per core; time = slowest worker (%.1f s, %.1f s with "
                      "process start-up and input generation)" % (n, tsteps, inner, wall)}


def cpu_reference_throughput(steps, warmup):
    """Times the reference's CPU path on all host cores (one process per core, independent
    chains, because the reference itself is single-threaded).  Returns (value, info dict)."""
    import multiprocessing as mp
    import build_ref
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    have_ref = build_ref.load("sv", 1024, NOBS, LAG) is not None
    ctx = mp.get_context("fork")
    if have_ref:
        n, kind, fn = 1024, "reference", _ref_worker
        make = lambda k: [(1000 * k + w, 1) for w in range(cores)]   # noqa: E731
    else:
        n, kind, fn = 16384, "port", _port_worker
        make = lambda k: [(1000 * k + w, n) for w in range(cores)]   # noqa: E731
    times = []
    with ctx.Pool(cores) as pool:
        for k in range(warmup + steps):
            t0 = time.perf_counter()
            pool.map(fn, make(k))
            dt = time.perf_counter() - t0
            if k >= warmup:
                times.append(dt)
    per_step = float(np.mean(times))
    value = cores * n * T_STEPS / per_step
    info = {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": "%s flps_sv_corr (hess=0), T=%d, N=%d, one independent evaluation per core "
                      "per step (N=2^20 is infeasible on the reference: O(T^2 N) ancestry copies)"
                      % ("compiled reference (oracle/_ref)" if have_ref else "oracle port", T_STEPS, n)}
    return value, per_step, info


def run_reference_arm(args, rank, world):
    """The CPU arm on the SAME config as ours (N = --particles, hess = 0): the reference's algorithm restated
    with O(T N) ancestry (oracle/pmmh_oracle.c, bit-exact against the compiled reference where that runs) on all
    host cores, one independent evaluation per core, each step a bounded sample of `--port-steps` time steps of
    the T = 1000 series.  The compiled reference itself (oracle/_ref) cannot run this config (O(T^2 N) ancestry
    copies, stack arrays); its number at N = 1024, its feasible size, is reported beside it."""
    if rank != 0:
        return
    import multiprocessing as mp
    n = args.particles
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cores = min(cores, 32)
    ctx = mp.get_context("fork")
    times = []
    with ctx.Pool(cores) as pool:
        for k in range(args.warmup + args.steps):
            res = pool.map(_port_sample_worker, [(1000 * k + w, n, args.port_steps) for w in range(cores)])
            if k >= args.warmup:
                times.append(max(r[0] for r in res))
    per_step = float(np.mean(times))
    value = cores * n * args.port_steps / per_step
    info = {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "oracle port (O(T N) restatement of flps_sv_corr, hess=0) at N=%d, %d of the %d time steps per "
                      "step, one independent evaluation per core (time = slowest worker)" % (n, args.port_steps, T_STEPS)}
    extra = None
    try:
        v2, _, info2 = cpu_reference_throughput(1, 0)
        extra = info2
    except Exception as e:   # reported
        extra = {"error": str(e)[:200]}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "sv_flps_T1000_N2^20_grad" if n == (1 << 20) else "sv_flps_T1000_N%d_grad" % n,
                   "T": T_STEPS, "N": n, "lag": LAG, "compute_hessian": 0,
                   "reference_sample": info["sample"]},
        "cpu_baseline": info,
        "cpu_baseline_compiled_reference": extra,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm
class BenchSVModel(object):
    """Minimal model object with the attributes the estimator reads (the reference's
    StochasticVolatilityModel, models/stochastic_volatility.py, stays ordinary Python)."""
    short_name = 'sv'

    def __init__(self, obs, params):
        self.obs = np.asarray(obs, dtype=np.float64).reshape(-1, 1)
        self.no_obs = self.obs.shape[0] - 1
        self.params = dict(zip(('mu', 'phi', 'sigma_v', 'rho'), [float(p) for p in params]))
        self.no_params = 4
        self.params_to_estimate = ('mu', 'phi', 'sigma_v', 'rho')
        self.params_to_estimate_idx = np.arange(4)
        self.using_gradients = True
        self.using_hessians = False

    def get_all_params(self):
        return np.array([self.params[k] for k in self.params])

    def log_prior_gradient(self):
        return {k: 0.0 for k in self.params}

    def log_prior_hessian(self):
        return {k: 0.0 for k in self.params}


def parity_at_shape(obs_h, params_t, rvr, u, n, psteps, dev):
    """The CUDA path against the oracle on the bench inputs themselves: the first `psteps` time steps
    of the headline problem (same N, same u).  Ancestors / sorted generations are compared at every
    step, the estimates to fp64 tolerances.  Also ties the full-length run to the prefix (filtered
    means are causal)."""
    import torch
    import oracle
    from pmmh_qn_b200 import kernels as K
    nobs = psteps + 1
    u_p = u[0, :nobs].contiguous()
    rvr_p = rvr[0, :nobs].contiguous()
    obs_p = torch.from_numpy(obs_h[:nobs].copy()).to(dev)
    out = K.flps_sv_corr(obs_p, params_t, rvr_p.reshape(1, nobs), u_p.reshape(1, nobs, n), lag=LAG,
                         compute_hessian=False, store_history=True)
    torch.cuda.synchronize()
    u_host = u_p.cpu().numpy()
    rvp = np.ascontiguousarray(u_host.T).reshape(-1)          # rvp[i + j * nobs]
    del u_host
    t0 = time.perf_counter()
    ref = oracle.flps_sv_corr(obs_h[:nobs].copy(), np.array(PARAMS), rvr_p.cpu().numpy(), rvp, n, LAG, 0, dumps=True)
    oracle_s = time.perf_counter() - t0
    A = out["A"][0].cpu().numpy()
    X = out["X"][0].cpu().numpy()
    mism = int(np.sum(np.any(A[1:] != ref["A"][1:], axis=1)))
    first = None
    if mism:
        first = int(np.argmax(np.any(A[1:] != ref["A"][1:], axis=1))) + 1
    ll = float(out["log_like"][0])
    g = out["gradient"][0].cpu().numpy()
    gref = np.asarray(ref["gradient"])
    d = out["diag"][0].tolist()
    return {"against": "oracle/pmmh_oracle.c (restates stochastic_volatility.pyx:205-655), same inputs as the timed run",
            "N": n, "time_steps": psteps, "kernel": KERNEL_NAMES.get(int(d[6]), "?"),
            "generations_mismatched": mism, "first_mismatch_step": first,
            "x_max_rel": float(np.max(np.abs(X - ref["X"])) / max(1e-300, np.max(np.abs(ref["X"])))),
            "ll_rel": abs(ll - ref["log_like"]) / abs(ref["log_like"]),
            "grad_rel": float(np.max(np.abs(g - gref)) / max(1e-300, np.max(np.abs(gref)))),
            "filt_rel": float(np.max(np.abs(out["filt"][0].cpu().numpy() - ref["filt"])) /
                              max(1e-300, np.max(np.abs(ref["filt"])))),
            "near_ties": int(d[0]), "soft_ties": int(d[4]) if int(d[6]) == 5 else None,
            "tie_note": "near_ties: decisions within 64 ulp of a cumulative-weight tie; soft_ties: decisions closer than "
                        "the bound on sequential-vs-parallel summation differences -- only those can pick another "
                        "ancestor than the reference (measured at T = 1000: profiles/r2_parity_full_N2^20_T1000.json)",
            "status": int(d[2]), "oracle_seconds": oracle_s,
            "tolerances": {"ancestors": "bit-exact", "ll_rel": 1e-10, "grad_rel": 1e-9, "filt_rel": 1e-10}}


def count_launches(fn):
    """Kernel launches of one call of fn(), counted from a CUPTI activity trace (torch.profiler)."""
    import torch
    try:
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = {}
        for ev in prof.events():
            if str(getattr(ev, "device_type", "")).endswith("CUDA"):
                nm = ev.name
                if nm.startswith("Memcpy") or nm.startswith("Memset"):
                    continue
                names[nm] = names.get(nm, 0) + 1
        total = sum(names.values())
        top = sorted(names.items(), key=lambda kv: -kv[1])[:6]
        return total, [{"kernel": k[:80], "launches": v} for k, v in top]
    except Exception as e:   # reported
        return None, [{"error": str(e)[:160]}]


def timed_events(fn, reps, warm):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    return float(np.median(ts))


# the estimates pmmh_flps_sv_corr returns (its diagnostics counters and workspace are not results)
DUMP_KEYS = ("log_like", "filt", "smo", "gradient", "traj", "hess1", "hess2")


def dump_outputs(out, path):
    """Writes the estimates of one evaluation as float64 `<name>.npy` files under `path` (about 100 KB at
    T = 1000), so that two builds can be compared output for output on the same seeded inputs."""
    os.makedirs(path, exist_ok=True)
    for k in DUMP_KEYS:
        np.save(os.path.join(path, k + ".npy"), out[k].cpu().numpy().astype(np.float64))


def max_over_ranks(seconds, dev, dist):
    import torch
    if dist is None:
        return seconds
    tt = torch.tensor([seconds], dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    return float(tt.item())


def run_config4_chains(rank, world, dev, dist, peak):
    """BASELINE configs[3]: 1024 independent SV chains x N = 4096 particles, T = 1000, one chain batch
    per GPU (1024 / world chains on every rank, no collective) => strong scaling."""
    import torch
    import golden_inputs as gi
    from pmmh_qn_b200 import kernels as K
    n, nobs, btot = 4096, NOBS, 1024
    b = btot // world
    g = torch.Generator(device=dev)
    g.manual_seed(400 + rank)
    obs = torch.from_numpy(gi.sv_obs(nobs)).to(dev)
    base = torch.tensor(PARAMS, dtype=torch.float64, device=dev)
    params = (base + 0.01 * torch.randn((b, 4), dtype=torch.float64, device=dev, generator=g)).contiguous()
    u = torch.randn((b, nobs, n), dtype=torch.float64, device=dev, generator=g)
    rvr = torch.rand((b, nobs), dtype=torch.float64, device=dev, generator=g)
    ws = K.Workspace()
    out = {}
    for hess in (False, True):
        fn = lambda: K.flps_sv_corr(obs, params, rvr, u, lag=LAG, compute_hessian=hess, workspace=ws)  # noqa: E731
        if dist is not None:
            dist.barrier()
        t = max_over_ranks(timed_events(fn, 2, 1), dev, dist)
        steps = btot * n * (nobs - 1)
        byt = (192 if hess else 96)
        o = fn()
        out["hessian" if hess else "gradient"] = {
            "seconds": t, "value": steps / t, "unit": UNIT, "loglik_evals_per_sec": btot / t,
            "kernel": KERNEL_NAMES.get(int(o["diag"][0, 6]), "?"), "status_max": int(o["diag"][:, 2].max()),
            "roofline": {"bound": "hbm", "achieved": steps * byt / t / 1e9 / world, "peak": peak, "unit": "GB/s",
                         "frac": steps * byt / t / 1e9 / world / peak, "traffic": None,
                         "algorithmic_bytes_per_particle_step": byt, "note": "per GPU"}}
    del u
    torch.cuda.empty_cache()
    return {"workload": "sv_flps_1024chains_N4096_T1000", "chains": btot, "chains_per_gpu": b, "N": n, "T": nobs - 1,
            "scaling": "strong", "n_gpus": world, **out}


def run_config4_lockstep(rank, world, dev, dist, iters=3):
    """BASELINE configs[3] as an actual sampler run: 1024 / world correlated pseudo-marginal chains per GPU
    in lock-step (parameter/lockstep.py), N = 4096, T = 1000, u of every chain resident in HBM (two
    [B, NOBS, N] tensors), Crank-Nicolson proposals on the device, ONE batched smoother launch per MH
    iteration, accept / reject per chain on the host.  The chains are pmmh_qn_b200.parameter.cpmh
    .CorrelatedPMMH (the reference's samplers are not available on the GPU box; they run under the same
    front-end unchanged: tests/test_lockstep_reference.py)."""
    import torch
    import golden_inputs as gi
    from pmmh_qn_b200.parameter.cpmh import BatchedRVSState, CorrelatedPMMH, _ChainRVS
    from pmmh_qn_b200.parameter.lockstep import LockstepRunner
    from pmmh_qn_b200.state.particle_methods.batched import BatchedParticleMethodsCUDA
    n, btot = 4096, 1024
    b = btot // world
    obs_h = gi.sv_obs(NOBS)
    state = BatchedRVSState(b, NOBS, n, dev, sigma_u=0.05, seed=900 + rank)
    rs = np.random.RandomState(40 + rank)
    chains = []
    for k in range(b):
        model = BenchSVModel(obs_h, PARAMS)
        model.no_params_to_estimate = 4
        init = np.array(PARAMS) + np.array([0.02, 0.005, 0.01, 0.01]) * rs.normal(size=4)
        chains.append(CorrelatedPMMH(model, {'no_iters': iters + 1, 'no_burnin_iters': 0, 'initial_params': init,
                                             'step_size': 0.01, 'precond': (1.0, 0.01, 0.05, 0.05), 'drift': True,
                                             'rvs': _ChainRVS(state, k)}))
    backend = BatchedParticleMethodsCUDA(chains[0].model, no_particles=n)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    runner = LockstepRunner(chains, backend, seeds=[5000 + 1000 * rank + k for k in range(b)]).run()
    torch.cuda.synchronize()
    secs = max_over_ranks(time.perf_counter() - t0, dev, dist)
    evals = iters + 1                                   # the initial evaluation + one per iteration
    acc = float(np.mean([np.mean([c.state_history[i]['accepted'] for i in range(1, iters + 1)]) for c in chains]))
    ll = np.array([c.state_history[iters]['log_like'] for c in chains])
    del state, backend, runner, chains
    torch.cuda.empty_cache()
    return {"workload": "cpmh_lockstep_1024chains_N4096_T1000", "chains": btot, "chains_per_gpu": b, "N": n, "T": T_STEPS,
            "mh_iterations": iters, "seconds": secs, "value": btot * n * T_STEPS * evals / secs, "unit": UNIT,
            "chain_iterations_per_sec": btot * iters / secs, "batched_launches_per_gpu": evals,
            "mean_acceptance": acc, "log_like_mean": float(ll.mean()), "all_finite": bool(np.all(np.isfinite(ll))),
            "n_gpus": world, "scaling": "strong",
            "note": "end to end through the sampler front-end: per iteration and chain a Crank-Nicolson pass over "
                    "its u (device), the batched smoother launch, results to the host, accept / reject in Python "
                    "(one coroutine per chain); the kernel-only figure is config4_chains"}


def run_config1_re(dev, peak):
    """BASELINE configs[0]: random-effects importance sampler, 100 individuals x 100 samples; one
    evaluation and batches of independent evaluations (proposals) per launch."""
    import torch
    import golden_inputs as gi
    from pmmh_qn_b200 import kernels as K
    nobs = n = 100
    obs_r, par_r, rvr_r, rvp_r = gi.re_inputs(n, nobs, 0)
    obs = torch.from_numpy(obs_r).to(dev)
    rows = []
    for B in (1, 1024, 65536):
        g = torch.Generator(device=dev)
        g.manual_seed(B)
        params = torch.tensor(par_r, dtype=torch.float64, device=dev).repeat(B, 1).contiguous()
        rvr = torch.rand((B,), dtype=torch.float64, device=dev, generator=g)
        rvp = torch.randn((B, nobs * n), dtype=torch.float64, device=dev, generator=g)
        t = timed_events(lambda: K.importance_discrete(obs, params, rvr, rvp, nobs, n), 5, 2)
        byt = B * nobs * n * 8
        rows.append({"batch": B, "seconds": t, "evals_per_sec": B / t,
                     "roofline": {"bound": "hbm", "achieved": byt / t / 1e9, "peak": peak, "unit": "GB/s",
                                  "frac": byt / t / 1e9 / peak, "traffic": None,
                                  "algorithmic_bytes_per_eval": nobs * n * 8}})
    return {"workload": "re_importance_100x100", "kernel": "importance_discrete_kernel (aux_kernels.cu)", "rows": rows}


def run_config3_subsampling(rank, world, dev, dist, peak):
    """BASELINE configs[2]: correlated data-subsampling estimator, n = 11 M x 28 regressors row-sharded
    over the ranks, m = 550 000 (5 %): Crank-Nicolson + Phi + sort + stratified indices (redundant on
    every rank) + gather-reduce of the owned rows + ONE all-reduce of 1 + d + d^2 doubles."""
    import torch
    from pmmh_qn_b200 import kernels as K
    n, d, m = 11_000_000, 28, 550_000
    per = (n + world - 1) // world
    r0, r1 = min(n, rank * per), min(n, (rank + 1) * per)
    g = torch.Generator(device=dev)
    g.manual_seed(30 + rank)
    x = torch.randn((r1 - r0, d), dtype=torch.float64, device=dev, generator=g)
    g0 = torch.Generator(device=dev)
    g0.manual_seed(31)
    beta = 0.1 * torch.randn((d,), dtype=torch.float64, device=dev, generator=g0)
    y = (torch.rand((r1 - r0,), dtype=torch.float64, device=dev, generator=g) < torch.sigmoid(x @ beta)).to(torch.float64)
    u = torch.randn((m,), dtype=torch.float64, device=dev, generator=g0)     # same u on every rank
    ws1, ws2 = K.Workspace(), K.Workspace()
    res = {}
    for hess in (False, True):
        def fn():
            un = K.crank_nicolson(u, 0.05, seed=1)
            idx = K.subsample_indices(un, n, workspace=ws1)
            o = K.logistic_loglike(x, y, idx, beta, compute_hessian=hess, row_begin=r0, row_end=r1, workspace=ws2)
            if dist is not None:
                dist.all_reduce(o, op=dist.ReduceOp.SUM)
            return o
        if dist is not None:
            dist.barrier()
        t = max_over_ranks(timed_events(fn, 5, 2), dev, dist)
        idx = K.subsample_indices(K.crank_nicolson(u, 0.05, seed=1), n, workspace=ws1)
        t_red = timed_events(lambda: K.logistic_loglike(x, y, idx, beta, compute_hessian=hess, row_begin=r0,
                                                        row_end=r1, workspace=ws2), 5, 2)
        byt = m * (8 * d + 12) / world
        res["hessian" if hess else "gradient"] = {
            "seconds": t, "rows_per_sec": m / t, "evals_per_sec": 1.0 / t, "gather_reduce_seconds_this_rank": t_red,
            "roofline": {"bound": "hbm", "achieved": byt / t_red / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": byt / t_red / 1e9 / peak, "traffic": None, "kernel": "logistic gather-reduce",
                         "algorithmic_bytes_per_row": 8 * d + 12}}
    del x, y
    torch.cuda.empty_cache()
    return {"workload": "logistic_subsampling_n11M_d28_m550000", "n_gpus": world, "scaling": "strong",
            "collective": "none (one rank)" if world == 1 else "one all_reduce(SUM) of %d doubles per evaluation (NCCL)" % (1 + d + d * d),
            **res}


def run_split_pf(args, rank, world, dev, dist):
    """Secondary measurement (not the headline): one SV smoother with N = 2^24 particles split over
    all ranks (pmmh_svsplit_* phases + NCCL all-gather / all-to-all per time step), T = 100,
    log-likelihood + gradient, u from a Philox stream.  Fixed N => strong scaling over --gpus."""
    import torch
    import golden_inputs as gi
    from pmmh_qn_b200 import kernels as K
    from pmmh_qn_b200.state.particle_methods import split as SP
    n, T = args.split_particles, args.split_steps
    nobs = T + 1
    obs = gi.sv_obs(nobs)
    comm = SP.DistComm() if dist is not None else SP.LocalComm(1)
    ph = SP.PhiloxRVS(seed=5, offset=0)
    rvr = K.norm_cdf(ph.resampling_normals(nobs, n, dev))
    secs, out = [], None
    try:
        for rep in range(2):
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = SP.run_split_smoother(comm, obs, np.array(PARAMS), n, LAG, rvr, philox=(5, 0), device=dev)
            e1.record()
            torch.cuda.synchronize()
            ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            if dist is not None:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            secs.append(float(ms.item()) * 1e-3)
    except Exception as e:     # reported, never silently replaced by another path
        return {"error": str(e)[:200]}
    return {"workload": "sv_flps_split_T%d_N2^%d_grad" % (T, int(np.log2(n))), "N": n, "T": T, "lag": LAG,
            "value": n * T / secs[-1], "unit": UNIT, "seconds": secs[-1], "scaling": "strong",
            "n_gpus": world, "log_like": float(out["log_like"].item()),
            "near_ties_rank0": int(out["diag"][0]), "status": int(out["diag"][2]),
            "max_particles_per_rank": int(out["counts"].max()),
            "exchange": "none (one rank, record variant: faster than path storage from N = 2^23 on)" if world == 1 else
                        "per step: all_gather 32 B + all_gather 16 KB + all_to_all of the 80-byte records that cross ranks (NCCL; the ones "
                        "that stay are packed straight into the receive buffer)"}


def run_ours(args, rank, world, local_rank):
    import torch
    import golden_inputs as gi
    from pmmh_qn_b200 import ParticleMethodsCUDA, kernels as K

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    n = args.particles
    obs_h = gi.sv_obs(NOBS)
    obs = torch.from_numpy(obs_h).to(dev)
    params = torch.tensor([PARAMS], dtype=torch.float64, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    # device-resident inputs (8.4 GB of u >> 126 MB of L2: nothing survives between steps)
    u = torch.randn((1, NOBS, n), dtype=torch.float64, device=dev, generator=g)
    rvr = torch.rand((1, NOBS), dtype=torch.float64, device=dev, generator=g)
    ws = K.Workspace()

    def step():
        return K.flps_sv_corr(obs, params, rvr, u, lag=LAG, compute_hessian=False, workspace=ws)

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        out = step()
    sync_all()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    e_all0 = torch.cuda.Event(enable_timing=True)
    e_all1 = torch.cuda.Event(enable_timing=True)
    e_all0.record()
    for k in range(args.steps):
        ev[k][0].record()
        out = step()
        ev[k][1].record()
    e_all1.record()
    sync_all()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    total_ms = e_all0.elapsed_time(e_all1)
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    if dist is not None:
        tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        total_ms = float(tt.item())
    ms_per_step = total_ms / args.steps
    value = world * n * T_STEPS / (ms_per_step * 1e-3)
    ll = float(out["log_like"][0])
    diag = out["diag"][0].tolist()

    # ---- the same workload on the other implementation of the path (not the headline): the
    # persistent exchange kernel (pmmh_sv_set_algorithm(2)) when the headline ran on the streaming
    # kernels, and the other way round
    alt = None
    alt_alg = 5 if int(diag[6]) == 5 else (2 if int(diag[6]) == 4 else 6)
    try:
        K.set_sv_algorithm(alt_alg)
        ws5 = K.Workspace()
        o5 = K.flps_sv_corr(obs, params, rvr, u, lag=LAG, compute_hessian=False, workspace=ws5)   # warm-up
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(2):
            o5 = K.flps_sv_corr(obs, params, rvr, u, lag=LAG, compute_hessian=False, workspace=ws5)
        a1.record()
        torch.cuda.synchronize()
        ms5 = a0.elapsed_time(a1) / 2
        alt = {"kernel": KERNEL_NAMES.get(int(o5["diag"][0, 6]), "?") + " (pmmh_sv_set_algorithm(%d))" % alt_alg,
               "ms_per_step": ms5,
               "value": n * T_STEPS / (ms5 * 1e-3), "unit": UNIT + " (this rank)",
               "log_like": float(o5["log_like"][0]), "status": int(o5["diag"][0, 2]),
               "rel_diff_log_like": abs(float(o5["log_like"][0]) - ll) / abs(ll)}
        del ws5, o5
    except Exception as e:   # reported, never silently replaced
        alt = {"error": str(e)[:200]}
    finally:
        K.set_sv_algorithm(0)

    # ---- the same workload with the Hessian branch (SURVEY 8a row a11: compute_hessian = 1, what the QN sampler's
    # 'hessian_estimate: kalman' style settings call), automatic kernel selection: the grid kernel's second
    # instantiation.  Algorithmic bytes per particle-step: the 96 B of the gradient path + 64 B (cumulative alpha
    # written next to the record and read back by the children and by the descendants lag - 2 steps later)
    with_hessian = None
    try:
        wsh = K.Workspace()
        oh = K.flps_sv_corr(obs, params, rvr, u, lag=LAG, compute_hessian=True, workspace=wsh)   # warm-up
        torch.cuda.synchronize()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        for _ in range(2):
            oh = K.flps_sv_corr(obs, params, rvr, u, lag=LAG, compute_hessian=True, workspace=wsh)
        h1.record()
        torch.cuda.synchronize()
        msh = h0.elapsed_time(h1) / 2
        with_hessian = {"kernel": KERNEL_NAMES.get(int(oh["diag"][0, 6]), "?"), "ms_per_step": msh,
                        "value": n * T_STEPS / (msh * 1e-3), "unit": UNIT + " (this rank)",
                        "status": int(oh["diag"][0, 2]),
                        "rel_diff_log_like": abs(float(oh["log_like"][0]) - ll) / abs(ll),
                        "hess1_trace": float(oh["hess1"][0].diagonal().sum()),
                        "roofline": {"bound": "hbm", "achieved": 160.0 * n * T_STEPS / (msh * 1e-3) / 1e9,
                                     "unit": "GB/s", "bytes_per_particle_step": 160}}
        del wsh, oh
    except Exception as e:   # reported, never silently replaced
        with_hessian = {"error": str(e)[:200]}

    # ---- launches of one step, counted (CUPTI activity trace of one extra, untimed step)
    launches_per_step, launch_top = count_launches(step)

    # ---- parity at the benchmarked shape: the oracle on the first time steps of the bench inputs
    parity = None
    if rank == 0 and world == 1 and args.parity_steps > 0:
        try:
            parity = parity_at_shape(obs_h, params, rvr, u, n, min(args.parity_steps, T_STEPS), dev)
            full_filt = out["filt"][0, :parity["time_steps"] + 1].cpu().numpy()
            pre = K.flps_sv_corr(torch.from_numpy(obs_h[:parity["time_steps"] + 1].copy()).to(dev), params,
                                 rvr[:, :parity["time_steps"] + 1].contiguous(),
                                 u[:, :parity["time_steps"] + 1].contiguous(), lag=LAG, compute_hessian=False)
            parity["full_run_filt_vs_prefix_rel"] = float(
                np.max(np.abs(full_filt - pre["filt"][0].cpu().numpy())) / max(1e-300, np.max(np.abs(full_filt))))
            del pre
        except Exception as e:   # reported, never hidden
            parity = {"error": str(e)[:300]}

    # ---- end to end through the public estimator API with HOST (pinned) buffers
    e2e_steps = max(1, args.e2e_steps)
    model = BenchSVModel(obs_h, PARAMS)
    est = ParticleMethodsCUDA(model, no_particles=n, fixed_lag=LAG, device=dev)
    rvs_pinned = torch.empty((NOBS, n + 1), dtype=torch.float64, pin_memory=True)
    rvs_pinned.copy_(torch.randn((NOBS, n + 1), dtype=torch.float64, device=dev, generator=g))
    rvs_np = rvs_pinned.numpy()
    del u
    torch.cuda.empty_cache()
    ok = est.smoother(model, rvs={'rvs': rvs_np})      # warm-up
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ok = est.smoother(model, rvs={'rvs': rvs_np}) and ok
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        tt = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item())
    e2e_value = world * n * T_STEPS * e2e_steps / e2e_s
    h2d = rvs_np.nbytes + (NOBS + 4 + NOBS) * 8
    d2h = (NOBS * 3 + 4 * NOBS + 1 + 32 + 8) * 8

    del rvs_pinned, rvs_np
    torch.cuda.empty_cache()

    # ---- end to end with the auxiliary variables RESIDENT on the device (the CPMH loop as it runs when u
    # never leaves HBM): Crank-Nicolson proposal with Philox normals into the spare slot, estimator call,
    # results to the host, accept / reject = slot swap
    e2e_dev = None
    try:
        from pmmh_qn_b200 import CorrelatedRVSState
        cst = CorrelatedRVSState.randn_particle(NOBS, n, dev, sigma_u=0.05, seed=77 + rank)
        okd = est.smoother(model, rvs={'rvs': cst.propose()})      # warm-up
        cst.accept()
        sync_all()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            prop = cst.propose()
            okd = est.smoother(model, rvs={'rvs': prop}) and okd
            if k % 2 == 0:
                cst.accept()
            else:
                cst.reject()
        torch.cuda.synchronize()
        e2e_dev_s = max_over_ranks(time.perf_counter() - t0, dev, dist)
        e2e_dev = {"value": world * n * T_STEPS * e2e_steps / e2e_dev_s, "unit": UNIT, "steps": e2e_steps, "ok": bool(okd),
                   "h2d_bytes_per_step": 32, "d2h_bytes_per_step": int(d2h),
                   "api": "CorrelatedRVSState.propose() -> ParticleMethodsCUDA.smoother(model, rvs={'rvs': handle}) "
                          "-> accept() / reject()",
                   "note": "u (2 x 8.4 GB slots) stays in HBM; per step: one Crank-Nicolson pass with Philox normals "
                           "(16 B per element), Phi of the resampling uniforms, the evaluation, results to the host"}
        del cst, prop
    except Exception as e:   # reported
        e2e_dev = {"error": str(e)[:200]}
    del est
    torch.cuda.empty_cache()
    peak, peak_src = measured_hbm_peak()

    # ---- the other BASELINE configs (secondary blocks, each with its own roofline)
    cfg1 = cfg3 = cfg4 = None
    if not args.no_configs:
        try:
            cfg4 = run_config4_chains(rank, world, dev, dist, peak)
        except Exception as e:
            cfg4 = {"error": str(e)[:200]}
        try:
            cfg4["lockstep_cpmh"] = run_config4_lockstep(rank, world, dev, dist)
        except Exception as e:
            if isinstance(cfg4, dict):
                cfg4["lockstep_cpmh"] = {"error": str(e)[:200]}
        try:
            cfg3 = run_config3_subsampling(rank, world, dev, dist, peak)
        except Exception as e:
            cfg3 = {"error": str(e)[:200]}
        if rank == 0:
            try:
                cfg1 = run_config1_re(dev, peak)
            except Exception as e:
                cfg1 = {"error": str(e)[:200]}

    # ---- BASELINE configs[4]: ONE particle filter split over the ranks (strong scaling, fixed N)
    split_line = None
    if not args.no_split:
        split_line = run_split_pf(args, rank, world, dev, dist)

    if rank == 0:
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
                tj = json.load(fh)
            args.traffic_bytes = float(tj["by_kernel"][str(int(diag[6]))]["dram_bytes_per_launch"])
        except Exception:
            pass
        achieved = n * T_STEPS * BYTES_PER_PARTICLE_STEP / (kern_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "sv_flps_T1000_N2^20_grad" if n == (1 << 20) else
                       "sv_flps_T1000_N%d_grad" % n,
                       "T": T_STEPS, "N": n, "lag": LAG, "compute_hessian": 0,
                       "per_gpu": "one independent evaluation per GPU per step (chain-batched sharding)",
                       "l2": "inputs larger than L2 (u = %.1f GB streamed once per step)" % (NOBS * n * 8 / 1e9)},
            "loglik_evals_per_sec": world / (ms_per_step * 1e-3),
            "log_like": ll, "near_ties": int(diag[0]), "status": int(diag[2]), "e2e_ok": bool(ok),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": args.traffic_bytes,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": n * T_STEPS * BYTES_PER_PARTICLE_STEP,
                         "kernel": KERNEL_NAMES.get(int(diag[6]), "sv_pf_kernel<false>"),
                         "kernel_ms": kern_ms,
                         "traffic_source": "ncu --set full capture of this kernel committed under profiles/ "
                                           "(profiles/traffic.json); not re-measured in this run",
                         "note": "kernel_ms = CUDA events around one pmmh_flps_sv_corr call on the launching "
                                 "stream (the persistent kernel plus its four small reduction / tail launches and "
                                 "the empty fallback pass); achieved = algorithmic bytes of the evaluation / that time"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                    "api": "ParticleMethodsCUDA.smoother(model, rvs={'rvs': pinned ndarray})",
                    "note": "host rvs -> pmmh_flps_sv_corr_streamed: the copy engine feeds the running grid kernel "
                            "in particle-major pieces of up to 256 time steps (2 KB rows, no layout kernel; pieces of ~0.3 x "
                            "the remaining steps towards the end so that the kernel ends a few ms after the last copy); the "
                            "kernel polls one flag per time step and re-lays every 32-byte sector (4 steps) of its particles "
                            "time-major once; bound by the host link (~52 GB/s); results read back to the host"},
            "gpu_launches": (launches_per_step * args.steps) if launches_per_step is not None else None,
            "gpu_launches_per_step": launches_per_step, "gpu_launches_top": launch_top,
            "gpu_launches_source": "CUPTI activity trace (torch.profiler) of one extra untimed step x steps",
        }
        if e2e_dev is not None:
            line["e2e_device_rvs"] = e2e_dev
        if parity is not None:
            line["parity"] = parity
        for key, blk in (("config1_re", cfg1), ("config3_subsampling", cfg3), ("config4_chains", cfg4)):
            if blk is not None:
                line[key] = blk
        if alt is not None:
            line["alt_kernel_same_workload"] = alt
        if with_hessian is not None:
            if "roofline" in with_hessian:
                with_hessian["roofline"].update(peak=peak, frac=with_hessian["roofline"]["achieved"] / peak)
            line["same_workload_with_hessian"] = with_hessian
        if split_line is not None:
            line["config5_split_pf"] = split_line
        if world == 1 and not args.no_cpu_baseline:
            _, _, info = cpu_reference_throughput(1, 0)
            line["cpu_baseline"] = info
            try:
                line["cpu_baseline_same_config"] = cpu_port_same_config(n, args.port_steps)
            except Exception as e:
                line["cpu_baseline_same_config"] = {"error": str(e)[:200]}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--particles", type=int, default=1 << 20)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--parity-steps", type=int, default=40,
                    help="time steps of the bench inputs re-run on the CPU oracle (0 = skip)")
    ap.add_argument("--port-steps", type=int, default=24,
                    help="time steps of the same-config CPU port sample (N = --particles on every core)")
    ap.add_argument("--no-configs", action="store_true", help="skip the config 1 / 3 / 4 blocks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-split", action="store_true", help="skip the config-5 split particle filter block")
    ap.add_argument("--split-particles", type=int, default=1 << 24)
    ap.add_argument("--split-steps", type=int, default=1000)
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram bytes per launch from the committed ncu capture (profiles/)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the estimates of the last timed step (rank 0) to DIR/<name>.npy (float64); "
                         "GPU path only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs covers the GPU path only (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.traffic_bytes is None:
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
                args.traffic_bytes = float(json.load(fh)["dram_bytes_per_launch"])
        except Exception:
            args.traffic_bytes = None
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
