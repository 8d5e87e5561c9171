"""Adaptive path tracing without a device: the C-ABI structs of rt_render_adaptive against gcc's layout, the
argument checks of CudaImageTracer.fire_all_rays_adaptive (ValueError before any device call) and the
`render` command refusing option combinations it cannot run."""
import ctypes
import os
import subprocess
import tempfile
import textwrap

import pytest
from click.testing import CliRunner

from pytracer_b200 import _abi, scenes
from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.imagetracer import CudaImageTracer
from pytracer_b200.main import cli
from pytracer_b200.pcg import PCG
from pytracer_b200.render import FlatRenderer, PathTracer

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
