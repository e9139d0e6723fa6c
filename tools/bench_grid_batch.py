#!/usr/bin/env python
"""Batches on the grid kernel (pmmh_flps_model_batch_corr: one team of G = ceil(N / 2048) CTAs per problem, waves of
floor(SMs / G) teams) against the other ways to evaluate the same B problems, T = 1000 (n_obs = 1001), lag 10:

  batch    the batch entry on the whole batch
  looped   B one-problem grid calls (flps_model_corr; with the Hessian flps_sv_corr at algorithm 6)
  auto     SV only: pmmh_flps_sv_corr's automatic choice on the whole batch (the exchange kernel for gradients, the
           general kernel with the Hessian)

Shapes: full waves at N = 2^14 .. 2^17 (B = floor(SMs / G): 18 / 9 / 4 / 2 on 148 SMs) and 2^16 x 16 (several waves);
SV and the linear Gaussian model with gradients, SV with the Hessian at 2^14 and 2^16.  Every arm is warmed up, the
arms alternate over --runs runs, each timed with CUDA events over --reps evaluations; the best run is reported
(ms per batch, particle-steps/s = B x N x T / time).  The script asserts that the batch and looped arms are
bit-identical.  One JSON line per shape, preceded by one line with the card, its power limit and clocks
(nvidia-smi --query-gpu, read-only); written to stdout and, with --out FILE, appended there.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import golden_inputs as gi  # noqa: E402
from pmmh_qn_b200 import _lib, kernels as K  # noqa: E402

KEYS = ("log_like", "filt", "smo", "gradient", "traj", "diag")


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
        return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().split(",")])) if r.stdout else None
    except (OSError, subprocess.SubprocessError):
        return None


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def looped(fn, batch, args):
    """B one-problem calls; the outputs stacked like a batch call's"""
    outs = [fn(*(t[b:b + 1] for t in args)) for b in range(batch)]
    return {k: torch.cat([o[k] for o in outs]) for k in outs[0] if not k.startswith("_")}


def with_algorithm(a, fn):
    K.set_sv_algorithm(a)
    try:
        return fn()
    finally:
        K.set_sv_algorithm(0)


def shape_record(model, n, batch, hess, nobs, lag, runs, reps, warm):
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(n + batch)
    u = torch.randn((batch, nobs, n), dtype=torch.float64, device=dev, generator=g)
    rvr = torch.rand((batch, nobs), dtype=torch.float64, device=dev, generator=g)
    sets = gi.SV_PARAM_SETS if model == 0 else gi.LG_PARAM_SETS
    params = np.array([sets[b % len(sets)] for b in range(batch)], dtype=np.float64)
    par = torch.from_numpy(params).to(dev)
    obs = torch.from_numpy(np.stack([gi.sv_obs(nobs) if model == 0 else gi.lg_obs(nobs, tuple(params[b]))
                                     for b in range(batch)])).to(dev)
    wb, wl, wa = K.Workspace(), K.Workspace(), K.Workspace()
    keys = KEYS + (("hess1", "hess2") if hess else ())
    arms = {"batch": lambda: K.flps_model_batch_corr(model, obs, par, rvr, u, lag=lag, compute_hessian=hess,
                                                     workspace=wb)}
    if hess:
        arms["looped"] = lambda: looped(lambda o, p, r, x: with_algorithm(6, lambda: K.flps_sv_corr(
            o, p, r, x, lag=lag, compute_hessian=True, workspace=wl)), batch, (obs, par, rvr, u))
    else:
        arms["looped"] = lambda: looped(lambda o, p, r, x: K.flps_model_corr(model, o, p, r, x, lag=lag, workspace=wl),
                                        batch, (obs, par, rvr, u))
    if model == 0:
        arms["auto"] = lambda: K.flps_sv_corr(obs, par, rvr, u, lag=lag, compute_hessian=bool(hess), workspace=wa)
    best, outs = {}, {}
    for name, fn in arms.items():   # warm-up of every arm
        for _ in range(warm):
            fn()
    torch.cuda.synchronize()
    for _ in range(runs):           # arms alternate
        for name, fn in arms.items():
            ms, outs[name] = timed(fn, reps)
            best[name] = min(best.get(name, ms), ms)
    for k in keys:
        assert torch.equal(outs["batch"][k], outs["looped"][k]), "batch and looped arms differ in %s" % k
    sm = K.device_info()[0]
    G = min((n + 2047) // 2048, sm)
    rec = {"model": ["sv", "lg", "lg_fa"][model], "hessian": bool(hess), "N": n, "B": batch, "G": G,
           "teams_per_wave": min(batch, sm // G), "n_obs": nobs, "lag": lag, "runs": runs, "reps": reps,
           "bit_identical_batch_looped": True}
    for name, ms in best.items():
        d = outs[name]["diag"].cpu().numpy()
        rec[name] = {"ms_per_batch": round(ms, 2), "particle_steps_per_s": float("%.4g" % (batch * n * (nobs - 1) /
                                                                                           (ms * 1e-3))),
                     "kernel": sorted(set(int(x) for x in d[:, _lib.DIAG_KERNEL])),
                     "status": sorted(set(int(x) for x in d[:, _lib.DIAG_STATUS]))}
    rec["speedup_batch_vs_looped"] = round(best["looped"] / best["batch"], 2)
    if "auto" in best:
        rec["speedup_batch_vs_auto"] = round(best["auto"] / best["batch"], 2)
    del u, rvr, wb, wl, wa
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nobs", type=int, default=1001)
    ap.add_argument("--lag", type=int, default=10)
    ap.add_argument("--runs", type=int, default=2)
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--quick", action="store_true", help="one shape per kind (a rehearsal)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_grid_batch.py needs a CUDA device")
    sm = K.device_info()[0]
    full = lambda n: max(1, sm // min((n + 2047) // 2048, sm))   # noqa: E731
    grad = [(n, full(n)) for n in (1 << 14, 1 << 15, 1 << 16, 1 << 17)] + [(1 << 16, 16)]
    shapes = [(0, n, b, 0) for n, b in grad] + [(1, n, b, 0) for n, b in grad] + \
             [(0, n, full(n), 1) for n in (1 << 14, 1 << 16)]
    if args.quick:
        shapes = [shapes[0], shapes[len(grad)], shapes[-1]]
    lines = [json.dumps({"gpu_state": gpu_state(), "sm_count": sm, "torch": torch.__version__})]
    print(lines[0], flush=True)
    for model, n, b, hess in shapes:
        lines.append(json.dumps(shape_record(model, n, b, hess, args.nobs, args.lag, args.runs, args.reps,
                                             args.warmup)))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
