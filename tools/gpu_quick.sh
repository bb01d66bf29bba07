#!/bin/bash
# quick check: the GPU tests that touch the train step + a short bench
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
python -m pytest tests -m gpu -q -p no:cacheprovider -x -k "trainer or cuda_graph or multilevel or wide or factored or activation or structure or fullsize or head or pool" > gpurun_out/r02_pytest_quick.log 2>&1
echo "pytest rc=$?"; grep -E "^(FAILED|ERROR)|passed|failed|Error" gpurun_out/r02_pytest_quick.log | head -20
python bench.py --no-cpu-baseline --no-diffpool --no-genconv > gpurun_out/r02_bench_quick.log 2>&1; echo "bench rc=$?"; tail -c 1200 gpurun_out/r02_bench_quick.log | head -c 600
