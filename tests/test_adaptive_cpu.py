"""Adaptive path tracing without a device: the C-ABI structs of rt_render_adaptive against gcc's layout, the
argument checks of CudaImageTracer.fire_all_rays_adaptive (ValueError before any device call), the
`render` command refusing option combinations it cannot run, and the host references the GPU error-map tests
compare with (tests/util.py batch_se2 and replay_adaptive)."""
import ctypes
import os
import subprocess
import tempfile
import textwrap

import numpy as np
import pytest
from click.testing import CliRunner

from pytracer_b200 import _abi, scenes
from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.imagetracer import CudaImageTracer
from pytracer_b200.main import cli
from pytracer_b200.pcg import PCG
from pytracer_b200.render import FlatRenderer, PathTracer
from util import batch_se2, replay_adaptive, same_partition

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DEMO_TXT = """
float clock(150)
material sky_material(diffuse(uniform(<0, 0, 0>)), uniform(<0.7, 0.5, 1>))
material ground_material(diffuse(checkered(<0.3, 0.5, 0.1>, <0.1, 0.2, 0.5>, 4)), uniform(<0, 0, 0>))
material sphere_material(specular(uniform(<0.5, 0.5, 0.5>)), uniform(<0, 0, 0>))
point_light([10, 10, 10], <1, 1, 1>, 1)
plane (sky_material, translation([0, 0, 100]) * rotation_y(clock))
plane (ground_material, identity)
sphere(sphere_material, translation([0, 0, 1]))
camera(perspective, rotation_z(30) * translation([-4, 0, 1]), 1.0, 1.0)
"""


def test_adaptive_struct_layouts_match_the_header():
    src = textwrap.dedent("""
        #include <stddef.h>
        #include <stdio.h>
        #include "rt_api.h"
        int main(void) {
          printf("%zu %zu %zu %zu %zu\\n", sizeof(rt_adaptive_params), sizeof(rt_adaptive_stats),
                 offsetof(rt_adaptive_stats, passes), offsetof(rt_adaptive_stats, pixels_in_pass),
                 offsetof(rt_adaptive_stats, overflow));
          return 0;
        }""")
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        sizes = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    S = _abi.rt_adaptive_stats
    assert [ctypes.sizeof(_abi.rt_adaptive_params), ctypes.sizeof(S), S.passes.offset, S.pixels_in_pass.offset,
            S.overflow.offset] == sizes


def _tracer(samples_per_side=4):
    world, camera = scenes.demo_scene()
    return CudaImageTracer(HdrImage(8, 6), camera, samples_per_side=samples_per_side), world


@pytest.mark.parametrize("case, kwargs, match", [
    ("flat renderer", {}, "path-tracing"),
    ("one sample per pixel", {"samples_per_side": 1}, "samples_per_side >= 2"),
    ("max not a multiple of S^2", {"max_samples_per_pixel": 24}, "multiple"),
    ("max below one pass", {"max_samples_per_pixel": 8}, "multiple"),
    ("negative target", {"target_error": -0.1}, "target_error"),
    ("NaN target", {"target_error": float("nan")}, "target_error"),
    ("zero floor", {"error_floor": 0.0}, "error_floor"),
    ("mega variant", {"variant": "mega"}, "warp"),
    ("fp64", {"precision": "f64"}, "warp"),
    ("two GPUs", {"gpus": 2}, "one device"),
])
def test_fire_all_rays_adaptive_checks_its_arguments_before_any_device_call(case, kwargs, match):
    kwargs = dict(kwargs)
    tracer, world = _tracer(kwargs.pop("samples_per_side", 4))
    renderer_kw = {k: kwargs.pop(k) for k in ("variant", "precision", "gpus") if k in kwargs}
    renderer = FlatRenderer(world) if case == "flat renderer" else PathTracer(world, pcg=PCG(45, 54), **renderer_kw)
    pcg_before = (tracer.pcg.state, renderer.pcg.state)
    with pytest.raises(ValueError, match=match):
        tracer.fire_all_rays_adaptive(renderer, **kwargs)
    assert renderer._scene is None  # nothing reached the device
    assert (tracer.pcg.state, renderer.pcg.state) == pcg_before


@pytest.mark.parametrize("args, message", [
    (["--algorithm", "flat", "--error-output", "e.pfm"], "pathtracing"),
    (["--samples-per-pixel", "1", "--error-output", "e.pfm"], "at least 4 samples"),
    (["--samples-per-pixel", "16", "--target-error", "0.05"], "go together"),
    (["--samples-per-pixel", "16", "--max-samples-per-pixel", "64"], "go together"),
    (["--samples-per-pixel", "16", "--target-error", "0.05", "--max-samples-per-pixel", "40"], "multiple"),
    (["--samples-per-pixel", "16", "--target-error", "-1", "--max-samples-per-pixel", "64"], "target-error"),
    (["--samples-per-pixel", "16", "--error-output", "e.pfm", "--error-floor", "0"], "error-floor"),
    (["--samples-per-pixel", "16", "--error-output", "e.pfm", "--gpus", "2"], "one GPU"),
    (["--samples-per-pixel", "16", "--error-output", "e.pfm", "--variant", "mega"], "warp"),
])
def test_render_command_refuses_adaptive_combinations_it_cannot_run(tmp_path, args, message):
    scene = tmp_path / "demo.txt"
    scene.write_text(DEMO_TXT)
    result = CliRunner().invoke(cli, ["render", "--width", "8", "--height", "6", "--pfm-output", str(tmp_path / "o.pfm"),
                                      "--png-output", str(tmp_path / "o.png"), *args, str(scene)])
    assert result.exit_code != 0, result.output
    assert "Error," in result.output and message in result.output, result.output
    assert not (tmp_path / "o.pfm").exists()


def test_batch_se2_is_the_documented_estimator():
    rng = np.random.default_rng(3)
    # one-sample batches (bpp >= L): the sample variance over L
    for L, bpp in ((4, 4), (9, 10), (16, 32), (25, 32)):
        x = rng.normal(2.0, 0.5, size=(7, 3, L))
        assert np.allclose(batch_se2(x, bpp), x.var(-1, ddof=1) / L, rtol=1e-12, atol=0), (L, bpp)
    # a layout given as labels equals the same layout given as bpp; the rounding bound is positive
    x = rng.normal(size=(5, 36))
    se2, bound = batch_se2(x, 32, bound=True)
    assert np.array_equal(se2, batch_se2(x, np.arange(36) % 32)) and (bound > 0).all()
    # unbiased for independent samples also where the batch sizes differ (n_b in {2, 1})
    for L, bpp in ((9, 8), (36, 32)):
        x = rng.normal(0.0, 1.5, size=(100_000, L))
        ratio = batch_se2(x, bpp).mean() / (1.5 ** 2 / L)
        print(f"L = {L}, bpp = {bpp}: mean SE^2 / (sigma^2 / L) = {ratio:.4f}")
        assert abs(ratio - 1.0) <= 0.01, (L, bpp, ratio)
    assert same_partition(np.arange(9) % 10, np.arange(9)) and not same_partition(np.arange(9) % 8, np.arange(9))
    assert same_partition([3, 3, 1, 1], [0, 0, 2, 2]) and not same_partition([0, 0, 1, 1], [0, 1, 0, 1])


def test_replay_adaptive_on_a_hand_made_example():
    """Three pixels, target 0.12, floor 0.01, three passes: pixel 0 is dark and stops after pass 0 because of the
    floor (without it e would be 1); pixel 1 misses the target after pass 0 and meets it after pass 1; pixel 2
    never does and stops at the pass limit.  NaN marks inputs of passes a pixel is not listed in."""
    nan = np.nan
    means = np.array([[[0.001] * 3, [0.5] * 3, [0.2] * 3],
                      [[nan] * 3, [0.7] * 3, [0.2] * 3],
                      [[nan] * 3, [nan] * 3, [0.2] * 3]], dtype=np.float32)[:, None]
    errs = np.array([[[0.001] * 3, [0.1, 0.0, 0.1], [0.2] * 3],
                     [[nan] * 3, [0.05, 0.0, 0.05], [0.2] * 3],
                     [[nan] * 3, [nan] * 3, [0.2] * 3]], dtype=np.float32)[:, None]
    r = replay_adaptive(means, errs, 0.12, 0.01, 3)
    assert r["passes"].tolist() == [[1, 2, 3]] and r["pixels_in_pass"] == [3, 2, 1] and not r["ambiguous"].any()
    f = np.float32
    assert np.array_equal(r["mean"][0, :, 0], [f(0.001), (f(0.5) + f(0.7)) / f(2), ((f(0.2) + f(0.2)) + f(0.2)) / f(3)])
    e1 = np.sqrt(f(0.1) ** 2.0 + f(0.05) ** 2.0) / 2
    assert np.allclose(r["err"][0, :, 0], [f(0.001), e1, np.sqrt(3 * f(0.2) ** 2.0) / 3], rtol=1e-12)
    assert r["err"][0, 1, 1] == 0.0
    # without the floor the dark pixel misses the target in every pass
    dark_m, dark_e = means.copy(), errs.copy()
    dark_m[:, 0, 0], dark_e[:, 0, 0] = 0.001, 0.001
    r = replay_adaptive(dark_m, dark_e, 0.12, 1e-6, 3)
    assert r["passes"].tolist() == [[3, 2, 3]] and r["pixels_in_pass"] == [3, 3, 2]
    # one pass, or a target no pixel misses: nothing is listed again
    assert replay_adaptive(means, errs, 0.12, 0.01, 1)["pixels_in_pass"] == [3]
    assert replay_adaptive(means, errs, float("inf"), 1e3, 3)["passes"].tolist() == [[1, 1, 1]]
    # a value at the target is ambiguous
    assert replay_adaptive(means, errs, 1.0, 1e-6, 3)["ambiguous"].tolist() == [[True, False, True]]
