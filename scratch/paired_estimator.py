"""The batch and the paired-strata error estimators side by side (rt_render_adaptive), on the current device.

    python scratch/paired_estimator.py OUT.json

1. Cost of the epilogue: config 3 (demo.txt 1920x1080, 64 spp), one error-map pass with each estimator,
   alternating in one process, and the plain render for reference.
2. Calibration: demo.txt 160x120, K = 16 seeds, 64 and 16 spp: the median over noisy values of
   mean(SE^2) / var(run means), and the fraction of values with |run - mean of runs| <= 3 SE.
3. Value at equal rays: demo.txt 1920x1080 and config 4 with accel="bvh" at 960x540, scored against a 4 096-spp
   uniform render as in scratch/adaptive_time.py: uniform 64 / 256 / 1 024 spp, then adaptive renders (16 spp per
   pass, at most 64 passes) at targets 0.05 / 0.02 / 0.01 with each estimator.
The card's name, power limit and clocks are read in the same run."""
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

EST = ("batch", "paired")
out = {}


def smi():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm,clocks_throttle_reasons.active",
                           "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()


out["gpu"] = smi()
print(out["gpu"], flush=True)
PT = dict(algorithm="pathtracing", num_of_rays=10, max_depth=3, rr_limit=3)

# ---- 1. cost of the epilogue
world, cam = scenes.demo_scene()
sc = DeviceScene(flatten_world(world))
p = make_params(1920, 1080, cam, samples_per_side=8, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **PT)
ms = {"plain": [], **{e: [] for e in EST}}
imgs = {}
for it in range(14):
    _, _, st = sc.render(p)
    if it >= 2:
        ms["plain"].append(st["kernel_ms"])
    for e in (EST if it % 2 == 0 else EST[::-1]):
        imgs[e], _, _, ast = sc.render_adaptive(p, 0.0, 1, estimator=e)
        if it >= 2:
            ms[e].append(ast["kernel_ms"])
ref, _, _ = sc.render(p)
out["c3_epilogue"] = dict(ms=ms, median={k: float(np.median(v)) for k, v in ms.items()},
                          range={k: [float(min(v)), float(max(v))] for k, v in ms.items()},
                          images_bit_identical=bool(all(np.array_equal(imgs[e], ref) for e in EST)), gpu_after=smi())
print("c3 epilogue:", out["c3_epilogue"]["median"], out["c3_epilogue"]["range"], out["c3_epilogue"]["images_bit_identical"], flush=True)

# ---- 2. calibration
fs_demo = flatten_world(world)
sc160 = DeviceScene(fs_demo)
out["calibration"] = {}
for S in (8, 4):
    runs, ses = [], {e: [] for e in EST}
    for k in range(16):
        pk = lambda: make_params(160, 120, cam, samples_per_side=S, aa_pcg=PCG(1000 + k, 7), pt_pcg=PCG(2000 + k, 9), **PT)
        for e in EST:
            mean, err, _, _ = sc160.render_adaptive(pk(), 0.0, 1, estimator=e)
            ses[e].append(err.astype(np.float64))
        runs.append(mean.astype(np.float64))
    runs = np.stack(runs)
    var_emp = runs.var(0, ddof=1)
    noisy = var_emp > 1e-12 * np.maximum(runs.mean(0) ** 2, 1e-6)
    res = {"noisy_values": int(noisy.sum())}
    for e in EST:
        se = np.stack(ses[e])
        ratio = float(np.median((se ** 2).mean(0)[noisy] / var_emp[noisy]))
        z = (runs - runs.mean(0)) / np.where(se > 0, se, np.inf)
        res[e] = dict(median_se2_over_var=ratio, within_3se=float((np.abs(z[:, noisy]) <= 3.0).mean()))
    out["calibration"][f"{S * S}spp"] = res
    print(f"calibration {S * S} spp:", res, flush=True)


# ---- 3. value at equal rays
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
        for e in EST:
            p = make_params(w, h, cam, samples_per_side=4, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw)
            img, _, samples, st = sc.render_adaptive(p, target, 64, estimator=e)
            p50, p99 = score(img, truth)
            res[f"adaptive_{target}_{e}"] = dict(rays=st["rays_closest"], ms=st["kernel_ms"], total_ms=st["total_ms"], p50=p50,
                                                 p99=p99, passes=st["passes"], hit_pass_limit=st["passes"] == 64,
                                                 pixels_in_pass=st["pixels_in_pass"], mean_spp=float(samples.mean()),
                                                 pixels_at_limit=int((samples == 64 * 16).sum()))
    for k, v in res.items():
        print(name, k, {a: b for a, b in v.items() if a != "pixels_in_pass"}, flush=True)
    return res


out["demo_1920x1080"] = study("demo 1920x1080", sc, 1920, 1080, cam, PT)
rs = scenes.random_spheres_scene(1024, 2024, 4, 20.0)
sc4 = DeviceScene(flatten_world(rs.world))
out["c4_bvh_960x540"] = study("c4 bvh 960x540", sc4, 960, 540, rs.camera, dict(PT, accel="bvh"))
out["gpu_end"] = smi()
with open(sys.argv[1], "w") as f:
    json.dump(out, f, indent=1)
