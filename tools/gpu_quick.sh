#!/bin/bash
# first contact of a new kernel with the GPU: short timeouts everywhere (a deadlocked kernel must not hold the box)
cd "$(dirname "$0")/.."
TAG=${1:-q}
mkdir -p gpurun_out
( timeout ${T1:-150} python -m pytest tests/test_gpu_ties.py tests/test_gpu_full_order.py -x -q -m gpu 2>&1 | tail -25 ) > gpurun_out/quick_tests_${TAG}.txt 2>&1
echo "rc=$?" >> gpurun_out/quick_tests_${TAG}.txt
( timeout ${T2:-150} python bench.py --config 3 --steps 3 --warmup 3 --no-cpu-baseline 2>&1 | tail -3 ) > gpurun_out/quick_bench_cfg3_${TAG}.log 2>&1
if [ -n "$FULL" ]; then ( time timeout 900 python -m pytest tests -x -q -m gpu ) > gpurun_out/pytest_gpu_${TAG}.txt 2>&1; tail -5 gpurun_out/pytest_gpu_${TAG}.txt; fi
if [ -n "$NCU" ]; then
timeout 300 ncu --set full --import-source on --clock-control none -k regex:score_select -c 1 -f -o gpurun_out/ncu_auc_${TAG} \
    python tools/run_once.py --config 3 --users 37888 --reps 1 > gpurun_out/ncu_auc_${TAG}.log 2>&1
fi
cat gpurun_out/quick_tests_${TAG}.txt | cut -c1-300; cat gpurun_out/quick_bench_cfg3_${TAG}.log | cut -c1-900
