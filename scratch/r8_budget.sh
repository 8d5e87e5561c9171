#!/bin/bash
# Round-8 batch for sample-budget rendering (profiles/r8_*), on one B200 with the in-tree library: the new GPU test
# file with its printed pass schedules, the whole suite, smoke(), a bench line, and scratch/budget_time.py (value
# against uniform sampling at equal samples, then the selection kernels under torch.profiler in a run of their own).
#   Usage: scratch/r8_budget.sh OUT_DIR
set -uo pipefail
cd "$(dirname "$0")/.."
OUT=${1:?usage: scratch/r8_budget.sh OUT_DIR}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv | tee $OUT/gpu.txt
python -m pytest tests/test_gpu_budget.py -q -s -p no:cacheprovider 2>&1 | tee $OUT/pytest_budget.txt | tail -8
python -m pytest tests -q -p no:cacheprovider 2>&1 | tail -15 | tee $OUT/pytest_all.txt
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -5 | tee $OUT/smoke.txt
python bench.py --gpus 1 --steps 5 --warmup 3 > $OUT/bench.json 2> $OUT/bench.err; tail -c 600 $OUT/bench.json
python scratch/budget_time.py study $OUT/budget_time.json 2>&1 | tee $OUT/budget_time.log
python scratch/budget_time.py profile $OUT/budget_profile.json 2>&1 | tail -40 | tee $OUT/budget_profile.log
