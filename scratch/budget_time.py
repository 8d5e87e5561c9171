"""Value of sample-budget rendering (rt_render_adaptive_budget) against uniform sampling at equal samples, on the
current device.

    python scratch/budget_time.py study   [OUT.json]
    python scratch/budget_time.py profile [OUT.json]

study: demo.txt at 1920x1080 and config 4 with accel="bvh" at 960x540, with the truth and seeds of
scratch/adaptive_time.py (4 096-spp uniform truth from PCG(7, 7) / PCG(8, 8), renders from PCG(42, 54) / PCG(45, 54)):
uniform 64 / 256 spp against budget means 64 / 256 spp (16 spp per pass, at most 1 024 spp, target 0), each with rays,
kernel and total ms, passes and the 50th / 99th percentile of |image - truth| / max(truth, 1e-2) over all values.
profile (a run of its own, torch.profiler with CUDA activities): device time of the combine and selection kernels of a
budget-256 render of demo.txt 1920x1080, in all and per selection.
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

mode = sys.argv[1] if len(sys.argv) > 1 else "study"
out = {"mode": mode}
out["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                            capture_output=True, text=True).stdout.strip()
print(out["gpu"], flush=True)
PT = dict(algorithm="pathtracing", num_of_rays=10, max_depth=3, rr_limit=3)


def score(img, truth):
    rel = np.abs(img.astype(np.float64) - truth) / np.maximum(truth, 1e-2)
    return float(np.percentile(rel, 50)), float(np.percentile(rel, 99))


def study(name, sc, w, h, cam, kw):
    res = {}
    truth, _, st = sc.render(make_params(w, h, cam, samples_per_side=64, aa_pcg=PCG(7, 7), pt_pcg=PCG(8, 8), **kw))
    truth = truth.astype(np.float64)
    res["truth"] = dict(spp=4096, ms=st["kernel_ms"], rays=st["rays_closest"])
    for spp_side in (8, 16):
        img, _, st = sc.render(make_params(w, h, cam, samples_per_side=spp_side, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw))
        p50, p99 = score(img, truth)
        res[f"uniform_{spp_side ** 2}"] = dict(rays=st["rays_closest"], ms=st["kernel_ms"], total_ms=st["total_ms"], passes=1,
                                               p50=p50, p99=p99, samples=st["samples"])
    for mean_spp in (64, 256):
        p = make_params(w, h, cam, samples_per_side=4, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw)
        img, _, samples, st = sc.render_budget(p, mean_spp * w * h, 64)
        p50, p99 = score(img, truth)
        res[f"budget_{mean_spp}"] = dict(rays=st["rays_closest"], ms=st["kernel_ms"], total_ms=st["total_ms"], p50=p50, p99=p99,
                                         passes=st["passes"], pixels_in_pass=st["pixels_in_pass"], samples=st["samples"],
                                         mean_spp=float(samples.mean()), max_spp=int(samples.max()),
                                         pixels_at_1024=int((samples == 1024).sum()))
    for k, v in res.items():
        print(name, k, {a: b for a, b in v.items() if a != "pixels_in_pass"}, flush=True)
    return res


if mode == "study":
    world, cam = scenes.demo_scene()
    sc = DeviceScene(flatten_world(world))
    out["demo_1920x1080"] = study("demo 1920x1080", sc, 1920, 1080, cam, PT)
    rs = scenes.random_spheres_scene(1024, 2024, 4, 20.0)
    sc4 = DeviceScene(flatten_world(rs.world))
    out["c4_bvh_960x540"] = study("c4 bvh 960x540", sc4, 960, 540, rs.camera, dict(PT, accel="bvh"))
else:
    import torch
    from torch.profiler import ProfilerActivity, profile

    world, cam = scenes.demo_scene()
    sc = DeviceScene(flatten_world(world))
    p = make_params(1920, 1080, cam, samples_per_side=4, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **PT)
    sc.render_budget(p, 64 * 1920 * 1080, 64)  # warm-up: module load, workspace
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, _, _, st = sc.render_budget(p, 256 * 1920 * 1080, 64)
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ("k_budget" in ev.name or "k_adaptive" in ev.name):
            key = ev.name.split("(")[0].replace("void ", "")
            k = kernels.setdefault(key, dict(calls=0, us=0.0))
            k["calls"] += 1
            k["us"] += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
    selections = kernels.get("k_budget_pick", {"calls": 0})["calls"] // 4
    sel_us = sum(v["us"] for k, v in kernels.items() if k.startswith("k_budget") or k in ("k_adaptive_offsets", "k_adaptive_scatter"))
    out["profile"] = dict(passes=st["passes"], pixels_in_pass=st["pixels_in_pass"], kernel_ms=st["kernel_ms"], selections=selections,
                          kernels=kernels, selection_us_total=sel_us, selection_us_per_pass=sel_us / max(selections, 1))
    print(json.dumps(out["profile"], indent=1), flush=True)
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as f:
        json.dump(out, f, indent=1)
