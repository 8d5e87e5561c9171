#!/bin/bash
# Round-7 batch for the SMALL path tracer (profiles/r7_*): parent build (scratch/v/parent.so, built from the parent
# commit's csrc with build_variant.sh) against this tree (scratch/v/new.so and the in-tree library) on one B200.
#   config 3, 4 and 5 outputs of both builds compared bit for bit; alternating kernel timings; a bench line per build;
#   resident blocks per SM of the c3 kernel; the drain-iteration mix (scratch/iteration_mix.py, scratch/v/mix.so);
#   the GPU suite and smoke().   Usage: scratch/r7_small.sh OUT_DIR
set -uo pipefail
cd "$(dirname "$0")/.."
OUT=${1:?usage: scratch/r7_small.sh OUT_DIR}
P=scratch/v/parent.so N=scratch/v/new.so
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv | tee $OUT/gpu.txt
for b in parent new; do
  lib=$P; [ $b = new ] && lib=$N
  for w in c3 c4 c5; do
    PYTRACER_B200_LIB=$lib python bench.py --workload $w --steps 2 --warmup 1 --no-extra --no-cpu-baseline --dump-outputs $OUT/dump_$b/$w > $OUT/dump_${b}_$w.json 2> $OUT/dump_${b}_$w.err
  done
done
python - "$OUT" <<'EOF' 2>&1 | tee $OUT/dump_compare.txt
import os, sys, numpy as np
o = sys.argv[1]
for w in ("c3", "c4", "c5"):
    for f in sorted(os.listdir(f"{o}/dump_parent/{w}")):
        a, b = np.load(f"{o}/dump_parent/{w}/{f}"), np.load(f"{o}/dump_new/{w}/{f}")
        print(w, f, a.shape, a.dtype, "array_equal", np.array_equal(a, b))
EOF
rm -rf $OUT/dump_parent $OUT/dump_new  # (the 4K frames would not fit the output directory)
python scratch/variants.py --workload c3 $P $N $P $N $P $N $P $N 2>&1 | tee $OUT/variants_c3.log
for b in parent new; do
  lib=$P; [ $b = new ] && lib=$N
  PYTRACER_B200_LIB=$lib python bench.py --gpus 1 --steps 5 --warmup 3 > $OUT/bench_$b.json 2> $OUT/bench_$b.err
  tail -c 600 $OUT/bench_$b.json
done
for b in parent new; do  # grid of the c3 kernel: the launcher sizes it to (resident blocks per SM) x SMs
  lib=$P; [ $b = new ] && lib=$N
  PYTRACER_B200_LIB=$lib python - <<'EOF' 2>&1 | tee -a $OUT/occupancy.txt
import os, torch, bench
from torch.profiler import profile, ProfilerActivity
from pytracer_b200.device import DeviceScene
world, camera, kw, desc, fpr, n_sph = bench.workload("c3")
sc = DeviceScene(world)
p = bench.build_params(kw, camera, accel="none", precision="auto", variant="auto")
img = torch.empty((p.height, p.width, 3), dtype=torch.float32, device="cuda")
sc.render_device(p, img.data_ptr()); sc.finish()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    sc.render_device(p, img.data_ptr()); sc.finish()
sms = torch.cuda.get_device_properties(0).multi_processor_count
for e in prof.events():
    if "k_pt_warp" in e.name:
        print(os.path.basename(os.environ["PYTRACER_B200_LIB"]), e.name[:60], "SMs", sms)
        break
prof.export_chrome_trace("/tmp/c3_trace.json")
import json
for ev in json.load(open("/tmp/c3_trace.json"))["traceEvents"]:
    if "k_pt_warp" in ev.get("name", ""):
        g = ev["args"].get("grid"); blk = ev["args"].get("block")
        print("  grid", g, "block", blk, "blocks per SM", g[0] / sms if g else None)
        break
EOF
done
python scratch/iteration_mix.py run $OUT/iteration_mix.json 2>&1 | tail -3
python -m pytest tests -m gpu -q -p no:cacheprovider 2>&1 | tail -15 | tee $OUT/pytest_gpu.txt
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -5 | tee $OUT/smoke.txt
