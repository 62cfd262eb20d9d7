#!/bin/bash
# round 2, call E: fp32 mode tests, fp32 floors, bench with the library comparator
mkdir -p gpurun_out
F='Warn\|Consider\|run_backward'
timeout 900 python -m pytest tests/test_iteration_gpu.py tests/test_round2_gpu.py tests/test_families.py -m gpu -q -s --tb=short -p no:cacheprovider -k "fp32" 2>&1 | grep -v "$F" > gpurun_out/pytest_e.log
grep -n "passed\|failed" gpurun_out/pytest_e.log | tail -3
grep -n "^FAILED\|deviations\|fp32 mode" gpurun_out/pytest_e.log | cut -c1-700
for cfg in "cond 0" "cond 0.5" "uncond 0"; do
  set -- $cfg
  timeout 900 python scripts/bf16_floor.py $1 $2 cuda fp32dev > gpurun_out/r02_fp32_floor_$1_g$2.json 2> gpurun_out/floor32_$1_$2.err
  cat gpurun_out/r02_fp32_floor_$1_g$2.json
done
timeout 900 python bench.py > gpurun_out/bench_e.json 2> gpurun_out/bench_e.err; tail -c 2500 gpurun_out/bench_e.json; tail -5 gpurun_out/bench_e.err
