#!/usr/bin/env python
"""Model id 8 (the SV model with the exact fixed-lag score, csrc/pf_model.cuh SvLeverageExact) against model 0 (the
reference's pairing) on the same inputs, alternating the two in every round.  Cases:

  grid       pmmh_flps_model_corr, one problem, N = 2^20, T = 1000 (n_obs = 1001), lag 10 (grid kernel)
  chain      pmmh_flps_model_corr, 1024 problems x N = 4096, n_obs = 1001, lag 10 (chain kernel)
  hess_grid  pmmh_flps_model_batch_corr with compute_hessian 1, one problem at the grid shape (model 0: the reference's
             Hessian branch, model 8: the generic one)
  hess_team  the same with 18 problems of N = 2^14 (team batch)

Each time is CUDA events around --reps evaluations after warm-up; ms_per_eval lists the rounds.  Prints one JSON line
per case with the card's name and power limit; --out FILE appends them there too.  Inputs: SV_PARAM_SETS[0] and
observations from golden_inputs.sv_obs, u and the resampling uniforms from a seeded torch generator.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import golden_inputs as gi  # noqa: E402
from bench_model_grid import power_limit, timed  # noqa: E402
from pmmh_qn_b200 import _lib, kernels as K  # noqa: E402

CASES = {   # name: (batch, N, hessian)
    "grid": (1, 1 << 20, 0),
    "chain": (1024, 4096, 0),
    "hess_grid": (1, 1 << 20, 1),
    "hess_team": (18, 1 << 14, 1),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--nobs", type=int, default=1001)
    ap.add_argument("--lag", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    card = torch.cuda.get_device_name(dev)
    plimit = power_limit()
    params = np.asarray(gi.SV_PARAM_SETS[0], dtype=np.float64)
    obs = torch.from_numpy(gi.sv_obs(args.nobs, params, seed=87655678)).to(dev)
    lines = []
    for name in args.cases.split(","):
        batch, n, hess = CASES[name]
        g = torch.Generator(device=dev)
        g.manual_seed(1234)
        u = torch.randn((batch, args.nobs, n), dtype=torch.float64, device=dev, generator=g)
        rvr = torch.rand((batch, args.nobs), dtype=torch.float64, device=dev, generator=g)
        par = torch.from_numpy(np.tile(params, (batch, 1))).to(dev)
        ws = {m: K.Workspace() for m in (0, 8)}

        def run(model):
            if hess:
                return K.flps_model_batch_corr(model, obs, par, rvr, u, lag=args.lag, compute_hessian=1,
                                               workspace=ws[model])
            return K.flps_model_corr(model, obs, par, rvr, u, lag=args.lag, workspace=ws[model])

        ms = {0: [], 8: []}
        outs = {}
        for _ in range(args.rounds):
            for model in (8, 0):
                t, outs[model] = timed(lambda: run(model), args.reps, args.warmup)
                ms[model].append(round(t, 3))
        d8, d0 = outs[8]["diag"].cpu().numpy(), outs[0]["diag"].cpu().numpy()
        same = all(torch.equal(outs[8][k], outs[0][k]) for k in ("filt", "log_like", "traj"))
        line = dict(case=name, batch=batch, n_particles=n, n_obs=args.nobs, lag=args.lag, compute_hessian=hess,
                    ms_per_eval_model8=ms[8], ms_per_eval_model0=ms[0],
                    ratio_best=round(min(ms[8]) / min(ms[0]), 4),
                    kernel=int(d8[0, _lib.DIAG_KERNEL]), status_model8=int(d8[:, _lib.DIAG_STATUS].max()),
                    status_model0=int(d0[:, _lib.DIAG_STATUS].max()), filter_outputs_identical=bool(same),
                    card=card, power_limit=plimit)
        print(json.dumps(line), flush=True)
        lines.append(line)
        del u, rvr, outs, ws
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
