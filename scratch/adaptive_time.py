"""Cost of the error map and value of noise-targeted passes (rt_render_adaptive), on the current device.

    python scratch/adaptive_time.py [OUT.json]

1. BASELINE config 3 (demo.txt 1920x1080, 64 spp): kernel time of rt_render and of the error-map kernel (one
   pass of rt_render_adaptive), alternating in one process.
2. demo.txt 1920x1080 and config 4 with accel="bvh" at 960x540: uniform renders of 64 / 256 / 1 024 spp and
   adaptive renders (16 spp per pass, at most 1 024) at three targets, each scored against a 4 096-spp uniform
   render: rays, ms and the 50th / 99th percentile of |image - truth| / max(truth, 1e-2) over all values.
The card's name and power limit are read in the same run."""
import json
import subprocess
import sys

import numpy as np

sys.path.insert(0, ".")
from pytracer_b200 import scenes  # noqa: E402
from pytracer_b200.device import DeviceScene  # noqa: E402
from pytracer_b200.flatten import flatten_world  # noqa: E402
from pytracer_b200.params import make_params  # noqa: E402
from pytracer_b200.pcg import PCG  # noqa: E402

out = {}
out["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                            capture_output=True, text=True).stdout.strip()
print(out["gpu"], flush=True)
PT = dict(algorithm="pathtracing", num_of_rays=10, max_depth=3, rr_limit=3)

# ---- 1. cost of the error map
world, cam = scenes.demo_scene()
sc = DeviceScene(flatten_world(world))
p = make_params(1920, 1080, cam, samples_per_side=8, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **PT)
plain, err = [], []
for it in range(12):
    _, _, st = sc.render(p)
    img, _, _, ast = sc.render_adaptive(p, 0.0, 1)
    if it >= 2:
        plain.append(st["kernel_ms"])
        err.append(ast["kernel_ms"])
ref, _, _ = sc.render(p)
out["c3_error_map"] = dict(plain_ms=plain, err_ms=err, plain_median=float(np.median(plain)), err_median=float(np.median(err)),
                           overhead=float(np.median(err) / np.median(plain) - 1), image_bit_identical=bool(np.array_equal(img, ref)))
print("c3 error map:", {k: v for k, v in out["c3_error_map"].items() if not isinstance(v, list)}, flush=True)


# ---- 2. value of adaptive sampling
def score(img, truth):
    rel = np.abs(img.astype(np.float64) - truth) / np.maximum(truth, 1e-2)
    return float(np.percentile(rel, 50)), float(np.percentile(rel, 99))


def study(name, sc, w, h, cam, kw):
    res = {}
    truth, _, st = sc.render(make_params(w, h, cam, samples_per_side=64, aa_pcg=PCG(7, 7), pt_pcg=PCG(8, 8), **kw))
    truth = truth.astype(np.float64)
    res["truth"] = dict(spp=4096, ms=st["kernel_ms"], rays=st["rays_closest"])
    for spp_side in (8, 16, 32):
        img, _, st = sc.render(make_params(w, h, cam, samples_per_side=spp_side, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw))
        p50, p99 = score(img, truth)
        res[f"uniform_{spp_side ** 2}"] = dict(rays=st["rays_closest"], ms=st["kernel_ms"], p50=p50, p99=p99)
    for target in (0.05, 0.02, 0.01):
        p = make_params(w, h, cam, samples_per_side=4, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw)
        img, _, samples, st = sc.render_adaptive(p, target, 64)
        p50, p99 = score(img, truth)
        res[f"adaptive_{target}"] = dict(rays=st["rays_closest"], ms=st["kernel_ms"], total_ms=st["total_ms"], p50=p50, p99=p99,
                                         passes=st["passes"], pixels_in_pass=st["pixels_in_pass"],
                                         mean_spp=float(samples.mean()))
    for k, v in res.items():
        print(name, k, {a: b for a, b in v.items() if a != "pixels_in_pass"}, flush=True)
    return res


out["demo_1920x1080"] = study("demo 1920x1080", sc, 1920, 1080, cam, PT)
rs = scenes.random_spheres_scene(1024, 2024, 4, 20.0)
sc4 = DeviceScene(flatten_world(rs.world))
out["c4_bvh_960x540"] = study("c4 bvh 960x540", sc4, 960, 540, rs.camera, dict(PT, accel="bvh"))
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        json.dump(out, f, indent=1)
