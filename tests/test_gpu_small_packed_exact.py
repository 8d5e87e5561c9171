"""The SMALL path tracer's packed FP32 arithmetic (fma.rn.f32x2 on paired transform rows and plane rows, see
closest_small in rt_warp.cuh) pinned bit for bit on scenes aimed at what packing can get wrong.

- exact zeros: an axis-aligned camera, translation-only transforms and planes whose inverse rows are mostly
  0, so that many products in the transform chains are +0 or -0 (a packed product must round like x * y,
  not like x * y + 0);
- rays parallel to a plane: a camera at a plane's height, mirror planes parallel to each other;
- spheres with a zero translation row, and non-uniformly scaled, rotated spheres;
- odd and even plane counts (planes are tested two at a time; an odd count pairs the last plane with zeros).

Each scene renders at 64 spp (one-pixel tasks) and 16 spp (multi-pixel tasks).  The fixtures are images,
per-pixel ray counts and the frame's ray count rendered on a B200 by the build before the packed forms
(tests/golden/make_golden_small_packed.py): any difference is a bug."""
import os

import numpy as np
import pytest

from pytracer_b200 import _abi
from pytracer_b200.device import DeviceScene
from pytracer_b200.flatten import flatten_camera, flatten_world
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG
from pytracer_b200.scene import (CheckeredPigment, Color, DiffuseBRDF, Material, PerspectiveCamera, Plane, SpecularBRDF,
                                 Sphere, Transformation, UniformPigment, Vec, rotation_x, rotation_z, scaling, translation,
                                 World)
from util import GOLDEN

W, H = 48, 32
BG = (0.2, 0.3, 0.4)


def _diffuse(c, emit=(0, 0, 0)):
    return Material(DiffuseBRDF(UniformPigment(Color(*c))), UniformPigment(Color(*emit)))


def _mirror(c):
    return Material(SpecularBRDF(UniformPigment(Color(*c))), UniformPigment(Color(0, 0, 0)))


def _checkered():
    return Material(DiffuseBRDF(CheckeredPigment(Color(0.3, 0.5, 0.1), Color(0.1, 0.2, 0.5), 4)), UniformPigment(Color(0, 0, 0)))


def _axis_aligned():
    """Camera along +x without rotation; a mirror floor and an emissive ceiling parallel to it, and spheres moved by
    translations only: every transform row but the translation column is 0 or 1."""
    world = World()
    world.add_shape(Sphere(translation(Vec(1, 0, 1)), _diffuse((0.8, 0.4, 0.2))))
    world.add_shape(Sphere(translation(Vec(0, -2, 0.5)) * scaling(Vec(0.5, 0.5, 0.5)), _mirror((0.7, 0.7, 0.7))))
    world.add_shape(Plane(Transformation(), _mirror((0.6, 0.6, 0.6))))
    world.add_shape(Plane(translation(Vec(0, 0, 4)), _diffuse((0.3, 0.3, 0.3), emit=(0.8, 0.7, 0.6))))
    return world, Transformation() * translation(Vec(-4, 0, 1))


def _grazing():
    """Camera at the height of the floor, so that primary rays run (nearly) parallel to it; a sphere centred at the
    origin (zero translation row); three planes, two of them parallel mirrors."""
    world = World()
    world.add_shape(Sphere(scaling(Vec(0.7, 0.7, 0.7)), _diffuse((0.7, 0.7, 0.3))))
    world.add_shape(Plane(Transformation(), _checkered()))
    world.add_shape(Plane(translation(Vec(0, 0, 2)), _mirror((0.8, 0.8, 0.8))))
    world.add_shape(Plane(rotation_x(90) * translation(Vec(0, 0, 3)), _diffuse((0.5, 0.2, 0.2), emit=(0.3, 0.3, 0.3))))
    return world, Transformation() * translation(Vec(-5, 0, 0))


def _stretched():
    """Non-uniformly scaled spheres, one rotated and one with a zero translation row, over one plane."""
    world = World()
    world.add_shape(Sphere(translation(Vec(0, -1, 1)) * rotation_z(30) * scaling(Vec(1.6, 0.4, 0.9)), _diffuse((0.8, 0.3, 0.3))))
    world.add_shape(Sphere(scaling(Vec(0.3, 2.0, 0.5)), _mirror((0.6, 0.6, 0.6))))
    world.add_shape(Sphere(translation(Vec(1, 1.5, 0.6)) * scaling(Vec(0.4, 0.4, 1.2)), _diffuse((0.2, 0.6, 0.9), emit=(1, 1, 1))))
    world.add_shape(Plane(translation(Vec(0, 0, -0.5)), _checkered()))
    return world, Transformation() * rotation_z(20) * translation(Vec(-5, 0, 1.5))


SCENES = {"axis_aligned": _axis_aligned, "grazing": _grazing, "stretched": _stretched}
# name: (samples_per_side, path-tracer parameters)
SETTINGS = {
    "spp64": (8, dict(num_of_rays=4, max_depth=5, rr_limit=2)),
    "spp16": (4, dict(num_of_rays=4, max_depth=5, rr_limit=2)),
}

_scenes = {}


def scene(name):
    if name not in _scenes:
        world, xf = SCENES[name]()
        flat = flatten_world(world)
        assert flat.n_shapes <= 16
        cam = flatten_camera(PerspectiveCamera(screen_distance=1.0, aspect_ratio=W / H, transformation=xf))
        _scenes[name] = (DeviceScene(flat), cam)
    return _scenes[name]


def render(name, setting):
    """What the fixture pins: the image, per-pixel ray counts and the frame's ray count."""
    sc, cam = scene(name)
    S, kw = SETTINGS[setting]
    p = make_params(W, H, cam, algorithm="pathtracing", samples_per_side=S, background=BG, aa_pcg=PCG(42, 54),
                    pt_pcg=PCG(45, 54), hit_mode=_abi.RT_HIT_RAY_COUNT, **kw)
    rgb, rays, st = sc.render(p, want_hit=True)
    assert st["overflow"] == 0
    return {"rgb": rgb, "rays": rays, "rays_closest": np.array([st["rays_closest"]], dtype=np.int64)}


def fixture_path(name):
    return os.path.join(GOLDEN, f"small_packed_{name}.npz")


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SETTINGS))
@pytest.mark.parametrize("name", list(SCENES))
def test_small_packed_is_exact(name, setting):
    want = np.load(fixture_path(name))
    got = render(name, setting)
    for key, value in got.items():
        ref = want[f"{setting}_{key}"]
        assert value.dtype == ref.dtype and np.array_equal(value, ref), (key, int((value != ref).sum()))
