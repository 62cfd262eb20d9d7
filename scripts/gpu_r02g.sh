#!/bin/bash
# round 2, call G: fp32 parity mode on exact fp32 FMA convolutions; 2-rank parity on the GPU
mkdir -p gpurun_out
F='Warn\|Consider\|run_backward'
timeout 1500 python -m pytest tests/test_iteration_gpu.py tests/test_round2_gpu.py tests/test_families.py tests/test_nrank_parity.py -m gpu -q -s --tb=short -p no:cacheprovider -k "fp32 or nrank or two_rank" 2>&1 | grep -v "$F" > gpurun_out/pytest_g.log
grep -n "passed\|failed" gpurun_out/pytest_g.log | tail -3
grep -n "^FAILED\|deviations\|fp32 mode\|2-rank\|Error" gpurun_out/pytest_g.log | cut -c1-700
