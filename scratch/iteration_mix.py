"""What the drain iterations of the SMALL path tracer do on config 3: a throw-away instrumented build, counters not in
the library's source.

    python scratch/iteration_mix.py build         # patches a copy of pytracer_b200/csrc, builds scratch/v/mix.so
    python scratch/iteration_mix.py run [OUT.json] # renders config 3 once with it (GPU) and prints the counts

Per warp and drain iteration (the primary rounds are not counted), from warp-uniform ballots:
  iterations, active lanes, iterations in which at least one lane pushes a record, pushing lanes, iterations in which
  every active lane is a leaf (depth == max_depth: no hit record, no scatter), iterations with a diffuse child.
Multiplied by static per-region instruction counts (scratch/sass_lines.py) they bound what a change to one region
can save.  The counters change the kernel's registers and schedule, so this build is for counting, not timing."""
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["drain_iterations", "active_lanes", "push_iterations", "pushing_lanes", "leaf_only_iterations", "diffuse_iterations"]

PATCH = [  # (file, anchor, text inserted after the anchor)
    ("rt_warp.cuh", "// SMALL: scenes of at most 8 spheres (demo.txt)", None),
    ("rt_warp.cuh", "  bool overflow = false;\n",
     "  unsigned long long mix[6] = {0, 0, 0, 0, 0, 0};\n"),
    ("rt_warp.cuh", "        // ---------------- pick this lane's ray\n",
     "        const bool mix_drain = !primary_phase;\n        bool mix_diffuse = false;\n"),
    ("rt_warp.cuh", "            if (((meta >> 5) & 1) == RT_BRDF_DIFFUSE) {\n", "              mix_diffuse = true;\n"),
    ("rt_warp.cuh", "        const int npush = __popc(pmask);\n",
     "        {\n"
     "          const unsigned act = __ballot_sync(FULL, active), inner = __ballot_sync(FULL, active && depth < a.max_depth);\n"
     "          const unsigned dif = __ballot_sync(FULL, active && mix_diffuse);\n"
     "          if (mix_drain) {\n"
     "            mix[0] += 1; mix[1] += __popc(act);\n"
     "            if (pmask) { mix[2] += 1; mix[3] += npush; }\n"
     "            if (inner == 0u) mix[4] += 1;\n"
     "            if (dif) mix[5] += 1;\n"
     "          }\n"
     "        }\n"),
    ("rt_warp.cuh", "  if (overflow) atomicExch(a.counters + CNT_OVERFLOW, 1ull);\n",
     "  if (lane == 0) for (int i = 0; i < 6; ++i) atomicAdd(&rt_mix[i], mix[i]);\n"),
]
PRELUDE = "__device__ unsigned long long rt_mix[6];\n"
READER = """
extern "C" int rt_mix_read(unsigned long long* out, int reset) {
  cudaError_t e = cudaMemcpyFromSymbol(out, rt_mix, sizeof(rt_mix));
  if (e == cudaSuccess && reset) {
    const unsigned long long z[6] = {0, 0, 0, 0, 0, 0};
    e = cudaMemcpyToSymbol(rt_mix, z, sizeof(z));
  }
  return (int)e;
}
"""


def build():
    tmp = tempfile.mkdtemp()
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tmp, "include"))
    src = os.path.join(tmp, "pytracer_b200", "csrc")
    shutil.copytree(os.path.join(ROOT, "pytracer_b200", "csrc"), src, ignore=shutil.ignore_patterns("build"))
    path = os.path.join(src, "rt_warp.cuh")
    text = open(path).read()
    for f, anchor, ins in PATCH:
        assert text.count(anchor) == 1, anchor
        text = text.replace(anchor, PRELUDE + anchor) if ins is None else text.replace(anchor, anchor + ins)
    open(path, "w").write(text)
    with open(os.path.join(src, "rt_kernels_f32.cu"), "a") as f:
        f.write(READER)
    subprocess.run(["bash", os.path.join(ROOT, "scratch", "build_variant.sh"), "mix", src], check=True)


def run(out=None):
    import ctypes
    lib_path = os.path.join(ROOT, "scratch", "v", "mix.so")
    os.environ["PYTRACER_B200_LIB"] = lib_path
    sys.path.insert(0, ROOT)
    import torch
    import bench
    from pytracer_b200.device import DeviceScene
    world, camera, kw, desc, fpr, n_sph = bench.workload("c3")
    sc = DeviceScene(world)
    p = bench.build_params(kw, camera, accel="none", precision="auto", variant="auto")
    img = torch.empty((p.height, p.width, 3), dtype=torch.float32, device="cuda")
    lib = ctypes.CDLL(lib_path)
    buf = (ctypes.c_ulonglong * 6)()
    sc.render_device(p, img.data_ptr()); sc.finish()
    assert lib.rt_mix_read(buf, 1) == 0
    sc.render_device(p, img.data_ptr()); st = sc.finish()
    assert lib.rt_mix_read(buf, 0) == 0
    r = dict(zip(NAMES, [int(x) for x in buf]))
    r["rays"] = int(st["rays_closest"])
    it = r["drain_iterations"]
    r["lanes_per_drain_iteration"] = r["active_lanes"] / it
    r["push_iteration_share"] = r["push_iterations"] / it
    r["pushing_lanes_per_push_iteration"] = r["pushing_lanes"] / max(r["push_iterations"], 1)
    r["leaf_only_share"] = r["leaf_only_iterations"] / it
    r["diffuse_iteration_share"] = r["diffuse_iterations"] / it
    r["gpu"] = torch.cuda.get_device_name(0)
    line = json.dumps(r)
    os.write(bench._REAL_STDOUT, (line + "\n").encode()) if hasattr(bench, "_REAL_STDOUT") else print(line)
    if out:
        open(out, "w").write(line + "\n")


if __name__ == "__main__":
    if sys.argv[1] == "build":
        build()
    else:
        run(sys.argv[2] if len(sys.argv) > 2 else None)
