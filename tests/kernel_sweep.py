"""Tiny renders through every kernel (run by test_every_kernel_at_tiny_sizes; also the script to put
under a memory / race checker: `compute-sanitizer python tests/kernel_sweep.py`)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from pytracer_b200 import scenes, _abi, tonemap
from pytracer_b200.device import DeviceScene
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG

def run(sc, cam, w, h, **kw):
    rgb, hit, st = sc.render(make_params(w, h, cam, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw), want_hit=True)
    assert np.isfinite(rgb).all() and st["overflow"] == 0
    return rgb

world, cam = scenes.demo_scene()
sc = DeviceScene(world)
for spp in (1, 2, 6):   # one-pixel tasks (36 strata), multi-pixel tasks, segmented accumulators
    run(sc, cam, 48, 27, algorithm="pathtracing", samples_per_side=spp, num_of_rays=4, max_depth=3, variant="warp")
run(sc, cam, 48, 27, algorithm="pathtracing", samples_per_side=2, num_of_rays=3, max_depth=3, variant="mega")
run(sc, cam, 48, 27, algorithm="pathtracing", samples_per_side=4, num_of_rays=3, max_depth=2, variant="warp",
    part_mode=_abi.RT_PART_SPP, part_rank=1, part_count=4)
rs = scenes.random_spheres_scene(150, 3, 4, 10.0, with_light=True)
big = DeviceScene(rs.world)
for accel in ("none", "bvh"):
    for algo in ("flat", "pointlight"):
        for prec in ("f32", "f64") + (("hybrid",) if accel == "none" else ()):
            for spp in (1, 2, 3):
                run(big, rs.camera, 40, 24, algorithm=algo, samples_per_side=spp, precision=prec, out_f64=(prec != "f32"), accel=accel)
    for variant in ("warp", "mega"):
        run(big, rs.camera, 40, 24, algorithm="pathtracing", samples_per_side=2, num_of_rays=3, max_depth=3, variant=variant, accel=accel)
# branching factors and depths at the edges of the work-stack sizing: N = 1 (a chain), deep trees, N larger
# than a warp, N beyond the multiply-shift division (1024); mega is the yardstick for the image mean
def lum(rgb):
    return float(((rgb.max(-1) + rgb.min(-1)) / 2).mean())

for n, depth, rr in ((1, 8, 3), (2, 6, 4), (40, 2, 2), (1100, 1, 3), (3, 0, 3)):
    for scene, camera, accels in ((sc, cam, ("none",)), (big, rs.camera, ("none", "bvh"))):
        ref = lum(run(scene, camera, 32, 18, algorithm="pathtracing", samples_per_side=3, num_of_rays=n, max_depth=depth, rr_limit=rr, variant="mega"))
        for accel in accels:
            got = lum(run(scene, camera, 32, 18, algorithm="pathtracing", samples_per_side=3, num_of_rays=n, max_depth=depth, rr_limit=rr,
                          variant="warp", accel=accel))
            assert abs(got - ref) <= 0.08 * ref + 1e-3, (n, depth, accel, got, ref)

# max_depth < 0: every sample is BLACK without tracing a ray (render.py:100-101); a depth the wavefront
# kernel's record format cannot hold (>= 1023): AUTO falls back to the depth-first kernel instead of failing
for variant in ("auto", "warp", "mega"):
    rgb, _, st = sc.render(make_params(16, 9, cam, algorithm="pathtracing", samples_per_side=2, num_of_rays=3, max_depth=-1, variant=variant))
    assert not rgb.any() and st["rays_closest"] == 0 and st["samples"] == 16 * 9 * 4
rgb, _, st = sc.render(make_params(16, 9, cam, algorithm="pathtracing", samples_per_side=1, num_of_rays=1, max_depth=2000, rr_limit=2))
assert st["variant_used"] == _abi.RT_VARIANT_MEGA and np.isfinite(rgb).all()

# error-map instantiations (rt_render_adaptive) at frames of one task, a partial last task and one row: one
# pass over the image, and three passes of which the later ones trace pixel lists
for scene, camera, accels in ((sc, cam, ("none",)), (big, rs.camera, ("none", "bvh"))):
    for accel in accels:
        for w, h in ((1, 1), (7, 3), (33, 1)):
            for spp in (2, 3):
                for passes in (1, 3):
                    p = make_params(w, h, camera, algorithm="pathtracing", samples_per_side=spp, num_of_rays=3, max_depth=3,
                                    accel=accel, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54))
                    mean, err, samples, st = scene.render_adaptive(p, 1e-6 if passes > 1 else 0.0, passes)
                    assert np.isfinite(mean).all() and np.isfinite(err).all() and (err >= 0).all() and st["overflow"] == 0
                    assert st["passes"] <= passes and ((samples >= spp * spp) & (samples <= passes * spp * spp)).all()

img = np.random.default_rng(1).random((37, 53, 3), dtype=np.float32) * 4
tonemap.average_luminosity(img)
tonemap.tone_map(img, 0.7, None, 1.0)
tonemap.tone_map(img, 0.7, 0.5, 2.2)
print("sanitize script done")
