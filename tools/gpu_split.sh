#!/bin/bash
# GPU check of the splitters: parity tests, timings beside the reference, and smoke()
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
timeout 420 python -m pytest tests/test_gpu_split.py -x -q -s 2>&1 | tail -25
echo "== timings"
for kind in all separated joined; do timeout 200 python tools/split_once.py --kind $kind 2>&1 | tail -1 | tee -a gpurun_out/split_once.jsonl; done
echo "== smoke"
timeout 200 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3
