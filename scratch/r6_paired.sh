#!/bin/bash
# Round-6 batch for the paired-strata error estimator (profiles/r6_*), on one B200 with the in-tree library:
# the new GPU test file with its printed bound ratios, the whole GPU suite, smoke(), a bench line, and
# scratch/paired_estimator.py (epilogue cost, calibration, value at equal rays for both estimators).
#   Usage: scratch/r6_paired.sh OUT_DIR
set -uo pipefail
cd "$(dirname "$0")/.."
OUT=${1:?usage: scratch/r6_paired.sh OUT_DIR}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv | tee $OUT/gpu.txt
python -m pytest tests/test_gpu_error_map_paired.py -q -s -p no:cacheprovider 2>&1 | tee $OUT/pytest_paired.txt | tail -5
python -m pytest tests -m gpu -q -p no:cacheprovider 2>&1 | tail -15 | tee $OUT/pytest_gpu.txt
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -5 | tee $OUT/smoke.txt
python bench.py --gpus 1 --steps 5 --warmup 3 > $OUT/bench.json 2> $OUT/bench.err; tail -c 600 $OUT/bench.json
python scratch/paired_estimator.py $OUT/paired_estimator.json 2>&1 | tee $OUT/paired_estimator.log
