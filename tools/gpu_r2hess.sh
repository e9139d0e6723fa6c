#!/bin/bash
# Hessian branch on the grid kernel: parity tests, then timings (grid kernel vs the general kernel)
mkdir -p gpurun_out
timeout 600 python -m pytest tests/test_gpu_sv_grid.py -x -q -k "hessian or vs_oracle or other_lags" 2>&1 | tail -15 | tee gpurun_out/r2hess_tests.log
for lg in 16 18 20; do
  echo "grid1024 hess logN $lg"; PMMH_PROBE_HESS=1 timeout 300 python tools/probe_alg.py 6 $lg 300 2 2>&1 | tail -1 | tee -a gpurun_out/r2hess_times.log
  echo "general hess logN $lg"; PMMH_PROBE_HESS=1 timeout 300 python tools/probe_alg.py 1 $lg 300 2 2>&1 | tail -1 | tee -a gpurun_out/r2hess_times.log
done
echo "grid nohess"; timeout 300 python tools/probe_alg.py 6 20 300 3 2>&1 | tail -1 | tee -a gpurun_out/r2hess_times.log
