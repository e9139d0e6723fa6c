#!/usr/bin/env python
"""pmmh_filter_model_corr (the filter alone) against pmmh_flps_model_corr (the fixed-lag smoother, lag 10) on the
same inputs, in one process, the two arms alternated:

  grid   one problem, N = 2^20, T = 1000 (n_obs = 1001), for each model id: SV (SV_PARAM_SETS[0], golden_inputs.sv_obs),
         linear Gaussian (LG_PARAM_SETS[0], golden_inputs.lg_obs) and the fully adapted filter (observations shifted
         by one, n_obs - 1 steps)
  chain  1024 problems x N = 4096, T = 1000, SV model (BASELINE config 4's shape)

Every call is timed alone with CUDA events: `--warmup` calls of each arm, then `--runs` rounds of (filter, smoother).
Per arm: ms per evaluation of each run, particle-steps/s of the faster run (problems x N x steps / time), and for the
filter its share of the HBM roofline at 44 B per particle-step (SURVEY 8(d): 7.7 TB/s, the B200 data sheet at 1000 W).
`identical`: log_like, filt, traj and diag of the two arms are bit-identical.  The card's name and power limit are
read in the same process.  Prints one JSON line; writes nothing unless --out FILE is given (the line is then
appended there as well).
"""
import argparse
import ctypes
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

HBM_BYTES_PER_S = 7.7e12
FILTER_BYTES_PER_PARTICLE_STEP = 44


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def ws_bytes(arm, nobs, n, lag, batch):
    lib, out = _lib.load(), ctypes.c_size_t()
    if arm == "filter":
        _lib.check(lib.pmmh_filter_model_workspace_bytes(nobs, n, batch, ctypes.byref(out)))
    else:
        _lib.check(lib.pmmh_flps_model_workspace_bytes(nobs, n, lag, batch, ctypes.byref(out)))
    return out.value


def timed_call(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def compare(model_id, obs, par, rvr, u, lag, runs, warmup):
    """filter and smoother on the same inputs, alternated; returns the case's record"""
    wf, ws = K.Workspace(), K.Workspace()
    arms = {"filter": lambda: K.filter_model_corr(model_id, obs, par, rvr, u, workspace=wf),
            "smoother": lambda: K.flps_model_corr(model_id, obs, par, rvr, u, lag=lag, workspace=ws)}
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    outs = {}
    for _ in range(runs):
        for k, fn in arms.items():
            t, outs[k] = timed_call(fn)
            ms[k].append(round(t, 3))
    batch, nobs, n = u.shape
    rec = {"batch": batch, "N": n, "n_obs": nobs}
    for k in arms:
        d = outs[k]["diag"].cpu().numpy()
        rate = batch * n * (nobs - 1) / (min(ms[k]) * 1e-3)
        rec[k] = {"ms_per_eval": ms[k], "particle_steps_per_s": float("%.4g" % rate),
                  "kernel": sorted(set(d[:, _lib.DIAG_KERNEL].tolist())),
                  "abandoned": int(np.sum(d[:, _lib.DIAG_STATUS] != 0)),
                  "workspace_bytes": ws_bytes(k, nobs, n, lag, batch)}
        if k == "filter":
            rec[k]["hbm_roofline_share"] = round(FILTER_BYTES_PER_PARTICLE_STEP * rate / HBM_BYTES_PER_S, 4)
    rec["identical"] = all(torch.equal(outs["filter"][k], outs["smoother"][k])
                           for k in ("log_like", "filt", "traj", "diag"))
    rec["log_like"] = float(outs["filter"]["log_like"][0])
    rec["filter_over_smoother"] = round(min(ms["filter"]) / min(ms["smoother"]), 4)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--nobs", type=int, default=1001)
    ap.add_argument("--lag", type=int, default=10)
    ap.add_argument("--chain-batch", type=int, default=1024)
    ap.add_argument("--chain-n", type=int, default=4096)
    ap.add_argument("--runs", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_filter_model.py needs a CUDA device")
    dev = torch.device("cuda:0")
    n, nobs, lag = args.n, args.nobs, args.lag
    res = {"lag": lag, "runs": args.runs, "warmup": args.warmup,
           "gpu": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    u = torch.randn((1, nobs, n), dtype=torch.float64, device=dev, generator=g)
    rvr = torch.rand((1, nobs), dtype=torch.float64, device=dev, generator=g)
    lg_par = np.array(gi.LG_PARAM_SETS[0])
    lg_obs = torch.from_numpy(gi.lg_obs(nobs, lg_par)).to(dev)
    lg_par = torch.from_numpy(lg_par).to(dev)
    sv_obs = torch.from_numpy(gi.sv_obs(nobs)).to(dev)
    sv_par = torch.from_numpy(np.array(gi.SV_PARAM_SETS[0])).to(dev)
    res["grid_sv"] = compare(_lib.MODEL_SV_LEVERAGE, sv_obs, sv_par, rvr, u, lag, args.runs, args.warmup)
    res["grid_lg"] = compare(_lib.MODEL_LINEAR_GAUSSIAN, lg_obs, lg_par, rvr, u, lag, args.runs, args.warmup)
    res["grid_lg_fa"] = compare(_lib.MODEL_LINEAR_GAUSSIAN_FA, lg_obs[1:].contiguous(), lg_par,
                                rvr[:, :nobs - 1].contiguous(), u[:, :nobs - 1].contiguous(), lag, args.runs,
                                args.warmup)
    del u, rvr
    torch.cuda.empty_cache()
    if args.chain_batch > 0:
        B, nc = args.chain_batch, args.chain_n
        uc = torch.randn((B, nobs, nc), dtype=torch.float64, device=dev, generator=g)
        rc = torch.rand((B, nobs), dtype=torch.float64, device=dev, generator=g)
        pc = torch.from_numpy(np.array([gi.SV_PARAM_SETS[b % len(gi.SV_PARAM_SETS)] for b in range(B)])).to(dev)
        res["chain_sv"] = compare(_lib.MODEL_SV_LEVERAGE, sv_obs, pc, rc, uc, lag, args.runs, args.warmup)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
