#!/usr/bin/env python
"""pmmh_flps_model_corr on the grid kernel at the headline shape: one problem, N = 2^20, T = 1000 (n_obs = 1001),
lag 10.  Nine cases, each timed with CUDA events over several evaluations after warm-up:

  lg_bootstrap  the linear Gaussian bootstrap filter (LG_PARAM_SETS[0], observations from golden_inputs.lg_obs)
  lg_fa         the same model as a fully adapted filter (observations shifted by one, n_obs - 1 steps)
  lg_fa_grad    the fully adapted filter with its fixed-lag gradient (model id 4, lg_fa's inputs)
  lg_fa_hess    model id 6 with its Hessian (pmmh_flps_model_batch_corr, batch 1, compute_hessian 1, lg_fa's inputs)
  lg_fa_hess0   the same call with compute_hessian 0 (it runs model 4's kernels)
  wave_fa_grad  a wave of --wave-batch problems of --wave-n particles, model 4 (pmmh_flps_model_batch_corr)
  wave_fa_hess  the same wave, model 6 with its Hessian
  sv_model      the SV model through pmmh_flps_model_corr (model id 0)
  sv_entry      pmmh_flps_sv_corr on the same SV inputs (algorithm 0: the grid kernel at this N)

--cases picks some of them, --rounds R runs the chosen cases in turn R times (alternating them; ms_per_eval is then the
list of the rounds, and the rate is of the fastest).  With lg_fa and lg_fa_grad both run, "fa_grad_shares_fa" says
whether lg_fa_grad's filt, smo, log_like, traj and diag equal lg_fa's bit for bit.
Prints one JSON line: ms per evaluation, particle-steps/s (N x steps / time), the card's name and power limit.
Writes nothing unless --out FILE is given (the line is then appended there as well).
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


def timed(fn, reps, warm):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--nobs", type=int, default=1001)
    ap.add_argument("--lag", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cases", default="lg_bootstrap,lg_fa,lg_fa_grad,sv_model,sv_entry")
    ap.add_argument("--wave-n", type=int, default=1 << 14)
    ap.add_argument("--wave-batch", type=int, default=18)
    ap.add_argument("--rounds", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_model_grid.py needs a CUDA device")
    dev = torch.device("cuda:0")
    n, nobs, lag = args.n, args.nobs, args.lag
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    u = torch.randn((1, nobs, n), dtype=torch.float64, device=dev, generator=g)
    rvr = torch.rand((1, nobs), dtype=torch.float64, device=dev, generator=g)
    lg_par = np.array(gi.LG_PARAM_SETS[0])
    lg_obs = torch.from_numpy(gi.lg_obs(nobs, lg_par)).to(dev)
    lg_par = torch.from_numpy(lg_par).to(dev)
    sv_obs = torch.from_numpy(gi.sv_obs(nobs)).to(dev)
    sv_par = torch.from_numpy(np.array(gi.SV_PARAM_SETS[0])).to(dev)
    fa_obs, fa_rvr, fa_u = lg_obs[1:].contiguous(), rvr[:, :nobs - 1].contiguous(), u[:, :nobs - 1].contiguous()
    ws = K.Workspace()
    K.set_sv_algorithm(0)
    names = args.cases.split(",")
    nw, bw = args.wave_n, args.wave_batch
    if any(c.startswith("wave_") for c in names):
        w_u = torch.randn((bw, nobs - 1, nw), dtype=torch.float64, device=dev, generator=g)
        w_rvr = torch.rand((bw, nobs - 1), dtype=torch.float64, device=dev, generator=g)
        w_par = lg_par.reshape(1, 4).repeat(bw, 1).contiguous()
    cases = {
        "lg_bootstrap": (nobs, lambda: K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN, lg_obs, lg_par, rvr, u, lag=lag,
                                                         workspace=ws)),
        "lg_fa": (nobs - 1, lambda: K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA, fa_obs, lg_par, fa_rvr, fa_u,
                                                      lag=lag, workspace=ws)),
        "lg_fa_grad": (nobs - 1, lambda: K.flps_model_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA_GRAD, fa_obs, lg_par, fa_rvr,
                                                           fa_u, lag=lag, workspace=ws)),
        "sv_model": (nobs, lambda: K.flps_model_corr(_lib.MODEL_SV_LEVERAGE, sv_obs, sv_par, rvr, u, lag=lag,
                                                     workspace=ws)),
        "sv_entry": (nobs, lambda: K.flps_sv_corr(sv_obs, sv_par, rvr, u, lag=lag, compute_hessian=False,
                                                  workspace=ws)),
        "lg_fa_hess": (nobs - 1, lambda: K.flps_model_batch_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA_HESS, fa_obs, lg_par,
                                                                 fa_rvr, fa_u, lag=lag, compute_hessian=1,
                                                                 workspace=ws)),
        "lg_fa_hess0": (nobs - 1, lambda: K.flps_model_batch_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA_HESS, fa_obs, lg_par,
                                                                  fa_rvr, fa_u, lag=lag, compute_hessian=0,
                                                                  workspace=ws)),
        "wave_fa_grad": (nobs - 1, lambda: K.flps_model_batch_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA_GRAD, fa_obs, w_par,
                                                                   w_rvr, w_u, lag=lag, workspace=ws)),
        "wave_fa_hess": (nobs - 1, lambda: K.flps_model_batch_corr(_lib.MODEL_LINEAR_GAUSSIAN_FA_HESS, fa_obs, w_par,
                                                                   w_rvr, w_u, lag=lag, compute_hessian=1,
                                                                   workspace=ws)),
    }
    res = {"N": n, "n_obs": nobs, "lag": lag, "reps": args.reps, "warmup": args.warmup,
           "gpu": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    times, outs = dict((k, []) for k in names), {}
    for _ in range(args.rounds):
        for name in names:
            ms, outs[name] = timed(cases[name][1], args.reps, args.warmup)
            times[name].append(round(ms, 3))
    for name in names:
        steps, out, ms = cases[name][0], outs[name], times[name]
        d = out["diag"][0].cpu().numpy()
        parts = nw * bw if name.startswith("wave_") else n
        res[name] = {"ms_per_eval": ms[0] if len(ms) == 1 else ms,
                     "particle_steps_per_s": float("%.4g" % (parts * (steps - 1) / (min(ms) * 1e-3))),
                     "kernel": int(d[_lib.DIAG_KERNEL]), "status": int(d[_lib.DIAG_STATUS]),
                     "log_like": float(out["log_like"][0])}
    if "lg_fa" in outs and "lg_fa_grad" in outs:
        res["fa_grad_shares_fa"] = all(torch.equal(outs["lg_fa"][k], outs["lg_fa_grad"][k])
                                       for k in ("filt", "smo", "log_like", "traj", "diag"))
    for a, b in (("lg_fa_grad", "lg_fa_hess"), ("lg_fa_hess0", "lg_fa_hess"), ("wave_fa_grad", "wave_fa_hess")):
        if a in outs and b in outs:   # model 6's outputs other than the Hessian are model 4's, bit for bit
            res["%s_shares_%s" % (b, a)] = all(torch.equal(outs[a][k], outs[b][k])
                                               for k in ("filt", "smo", "log_like", "gradient", "traj", "diag"))
    if any(c.startswith("wave_") for c in names):
        res["wave"] = {"N": nw, "batch": bw}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
