#!/bin/bash
mkdir -p gpurun_out
timeout 900 ncu --set full --import-source on --clock-control none -k regex:sv_grid_kernel -c 1 -f -o gpurun_out/r2d_grid python tools/probe_alg.py 6 20 100 1 > gpurun_out/r2d_ncu.log 2>&1
tail -3 gpurun_out/r2d_ncu.log; ls -la gpurun_out/*.ncu-rep
