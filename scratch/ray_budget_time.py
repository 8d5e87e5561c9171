"""Ray-budget rendering (rt_render_adaptive_rays) against uniform sampling and the sample-budget mode, on the current
device.

    python scratch/ray_budget_time.py study   [OUT.json]
    python scratch/ray_budget_time.py profile [OUT.json]
    python scratch/ray_budget_time.py errpass [OUT.json]   (also from a checkout of the parent build: counting off only)

study: demo.txt at 1920x1080 and config 4 with accel="bvh" at 960x540, with the truth, seeds and error metric of
scratch/budget_time.py (4 096-spp uniform truth from PCG(7, 7) / PCG(8, 8), renders from PCG(42, 54) / PCG(45, 54),
16 spp per pass, at most 1 024 spp, target 0): uniform 64 / 256 spp, the sample budget at means 64 / 256 spp, and the
ray budget at the rays uniform 64 / 256 spp traced in the same run; each with rays, kernel ms, passes, the largest
per-pixel spp and the 50th / 99th percentile of |image - truth| / max(truth, 1e-2) over all values.
profile (a run of its own, torch.profiler with CUDA activities): device time of the combine and selection kernels of a
ray-budget render of demo.txt 1920x1080 at the rays of uniform 256 spp, in all and per selection.
errpass: kernel time of one error-map pass (rt_render_adaptive with one pass: no ray counting; rt_render_adaptive_rays
with R = 0 and one pass: per-pixel ray counting), alternating in one process, on demo.txt 1920x1080 at 64 and 16 spp
and config 4 (bvh, 960x540) at 16 spp.
The card's name, power limit and max SM clock are read in the same run."""
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
MAX_PASSES = 1024 // 16


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
        res[f"uniform_{spp_side ** 2}"] = dict(rays=st["rays_closest"], ms=st["kernel_ms"], passes=1, max_spp=spp_side ** 2,
                                               p50=p50, p99=p99)
    p = make_params(w, h, cam, samples_per_side=4, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw)
    for spp in (64, 256):
        img, _, samples, st = sc.render_budget(p, spp * w * h, MAX_PASSES)
        p50, p99 = score(img, truth)
        res[f"samples_{spp}"] = dict(rays=st["rays_closest"], ms=st["kernel_ms"], passes=st["passes"], max_spp=int(samples.max()),
                                     mean_spp=float(samples.mean()), p50=p50, p99=p99)
        R = res[f"uniform_{spp}"]["rays"]
        img, _, samples, rays, st = sc.render_rays(p, R, MAX_PASSES)
        p50, p99 = score(img, truth)
        res[f"rays_{spp}"] = dict(ray_budget=R, rays=st["rays_closest"], overrun=st["rays_closest"] - R, ms=st["kernel_ms"],
                                  passes=st["passes"], max_spp=int(samples.max()), mean_spp=float(samples.mean()), p50=p50, p99=p99,
                                  max_pixel_rays=int(rays.max()), pixels_in_pass=st["pixels_in_pass"])
    for k, v in res.items():
        print(name, k, {a: b for a, b in v.items() if a != "pixels_in_pass"}, flush=True)
    return res


def errpass(name, sc, w, h, cam, kw, S, iters=10):
    p = make_params(w, h, cam, samples_per_side=S, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw)
    counting = hasattr(sc, "render_rays")
    off, on = [], []
    for it in range(iters + 2):
        _, _, _, st = sc.render_adaptive(p, 0.0, 1)
        if counting:
            _, _, _, _, rst = sc.render_rays(p, 0, 1)
        if it >= 2:
            off.append(st["kernel_ms"])
            if counting:
                on.append(rst["kernel_ms"])
    r = dict(off_ms=off, off_median=float(np.median(off)))
    if counting:
        r.update(on_ms=on, on_median=float(np.median(on)), on_over_off=float(np.median(on) / np.median(off)))
    print(name, {k: v for k, v in r.items() if not k.endswith("_ms")}, flush=True)
    return r


if mode == "study":
    world, cam = scenes.demo_scene()
    sc = DeviceScene(flatten_world(world))
    out["demo_1920x1080"] = study("demo 1920x1080", sc, 1920, 1080, cam, PT)
    rs = scenes.random_spheres_scene(1024, 2024, 4, 20.0)
    sc4 = DeviceScene(flatten_world(rs.world))
    out["c4_bvh_960x540"] = study("c4 bvh 960x540", sc4, 960, 540, rs.camera, dict(PT, accel="bvh"))
elif mode == "errpass":
    world, cam = scenes.demo_scene()
    sc = DeviceScene(flatten_world(world))
    out["demo_1920x1080_64spp"] = errpass("demo 1920x1080 64 spp", sc, 1920, 1080, cam, PT, 8)
    out["demo_1920x1080_16spp"] = errpass("demo 1920x1080 16 spp", sc, 1920, 1080, cam, PT, 4)
    rs = scenes.random_spheres_scene(1024, 2024, 4, 20.0)
    sc4 = DeviceScene(flatten_world(rs.world))
    out["c4_bvh_960x540_16spp"] = errpass("c4 bvh 960x540 16 spp", sc4, 960, 540, rs.camera, dict(PT, accel="bvh"), 4)
else:
    import torch
    from torch.profiler import ProfilerActivity, profile

    world, cam = scenes.demo_scene()
    sc = DeviceScene(flatten_world(world))
    _, _, st = sc.render(make_params(1920, 1080, cam, samples_per_side=16, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **PT))
    R = st["rays_closest"]
    p = make_params(1920, 1080, cam, samples_per_side=4, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **PT)
    sc.render_rays(p, R // 4, MAX_PASSES)  # warm-up: module load, workspace
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, _, _, _, st = sc.render_rays(p, R, MAX_PASSES)
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
    out["profile"] = dict(ray_budget=R, rays=st["rays_closest"], passes=st["passes"], pixels_in_pass=st["pixels_in_pass"],
                          kernel_ms=st["kernel_ms"], selections=selections, kernels=kernels, selection_us_total=sel_us,
                          selection_us_per_pass=sel_us / max(selections, 1))
    print(json.dumps(out["profile"], indent=1), flush=True)
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as f:
        json.dump(out, f, indent=1)
