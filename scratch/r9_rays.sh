#!/bin/bash
# Round-9 batch for ray-budget rendering (profiles/r9_*), on one B200 with the in-tree library: the new GPU test file
# with its printed pass schedules, the whole suite, smoke(), a bench line, the error-map pass with ray counting on and
# off against the parent build (a checkout of the parent commit with its library, at PARENT, alternating three times),
# and scratch/ray_budget_time.py study, then profile in a run of its own.
#   Usage: scratch/r9_rays.sh OUT_DIR [PARENT]
set -uo pipefail
cd "$(dirname "$0")/.."
OUT=${1:?usage: scratch/r9_rays.sh OUT_DIR [PARENT]}
PARENT=${2:-}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv | tee $OUT/gpu.txt
python -m pytest tests/test_gpu_ray_budget.py -q -s -p no:cacheprovider 2>&1 | tee $OUT/pytest_rays.txt | tail -8
python -m pytest tests -q -p no:cacheprovider 2>&1 | tail -15 | tee $OUT/pytest_all.txt
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -5 | tee $OUT/smoke.txt
python bench.py --gpus 1 --steps 5 --warmup 3 > $OUT/bench.json 2> $OUT/bench.err; tail -c 600 $OUT/bench.json
for i in 1 2 3; do
  if [ -n "$PARENT" ]; then (cd $PARENT && python "$OLDPWD/scratch/ray_budget_time.py" errpass "$OLDPWD/$OUT/errpass_parent_$i.json") 2>&1 | tee -a $OUT/errpass.log; fi
  python scratch/ray_budget_time.py errpass $OUT/errpass_new_$i.json 2>&1 | tee -a $OUT/errpass.log
done
python scratch/ray_budget_time.py study $OUT/ray_budget_time.json 2>&1 | tee $OUT/ray_budget_time.log
python scratch/ray_budget_time.py profile $OUT/ray_budget_profile.json 2>&1 | tail -40 | tee $OUT/ray_budget_profile.log
