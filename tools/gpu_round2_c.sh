#!/bin/bash
mkdir -p gpurun_out
timeout 600 python -m pytest tests/test_gpu_sv_grid.py -x -q -m gpu > gpurun_out/r2c_tests.log 2>&1; echo "tests(512) exit $?" >> gpurun_out/r2c_tests.log
grep -E "passed|failed|exit|Error|assert" gpurun_out/r2c_tests.log | head -20
for d in 1 4 7; do echo "dbg $d"; PMMH_GRID_DEBUG=$d timeout 200 python tools/phase_clocks_grid.py 20 300 2>&1 | grep -v "wait\|zero\|shift" | tee -a gpurun_out/r2c_dbg.log; done
