"""The SMALL path tracer (k_pt_warp with every scene table in shared memory: at most 8 spheres and 16 shapes)
pinned bit for bit across its shape-count range.

Six scenes, from 0 spheres + 1 plane to the largest SMALL scene (8 spheres + 8 planes), with uv-dependent
and image pigments and an emissive sphere, each at the settings that select the kernel's instantiations:
64 spp (one-pixel tasks, lane-private sums: ACC_REG), 16 spp (multi-pixel tasks), one ray per interaction
(the N = 1 work stack) and one pass of the error map (ERR).  The fixtures are images and per-pixel ray
counts rendered on a B200 by the build before the SMALL closest-hit walk was unrolled and the primary
jitter moved to a per-block jump table (tests/golden/make_golden_small.py), which are exact rewrites: any
difference is a bug."""
import os

import numpy as np
import pytest

from pytracer_b200 import _abi, scenes
from pytracer_b200.device import DeviceScene
from pytracer_b200.flatten import flatten_camera, flatten_world
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG
from pytracer_b200.scene import (CheckeredPigment, Color, DiffuseBRDF, ImagePigment, Material, PerspectiveCamera, Plane,
                                 SpecularBRDF, Sphere, Transformation, UniformPigment, Vec, rotation_x, rotation_y,
                                 rotation_z, scaling, translation, World)
from util import GOLDEN, demo_flat

W, H = 48, 32
BG = (0.2, 0.3, 0.4)


def _camera():
    return PerspectiveCamera(screen_distance=1.0, aspect_ratio=W / H,
                             transformation=Transformation() * rotation_z(20) * translation(Vec(-5, 0, 1.5)))


def _diffuse(c, emit=(0, 0, 0)):
    return Material(DiffuseBRDF(UniformPigment(Color(*c))), UniformPigment(Color(*emit)))


def _checkered():
    return Material(DiffuseBRDF(CheckeredPigment(Color(0.3, 0.5, 0.1), Color(0.1, 0.2, 0.5), 4)), UniformPigment(Color(0, 0, 0)))


def _one_plane():
    world = World()
    world.add_shape(Plane(Transformation(), _checkered()))
    return world


def _two_spheres():
    world = World()
    world.add_shape(Sphere(translation(Vec(0, -1, 1)), _diffuse((0.8, 0.4, 0.2))))
    world.add_shape(Sphere(translation(Vec(0, 1.2, 1)) * scaling(Vec(0.8, 0.8, 0.8)),
                           Material(SpecularBRDF(UniformPigment(Color(0.6, 0.6, 0.6))), UniformPigment(Color(0, 0, 0)))))
    return world


def _largest():
    """8 spheres + 8 planes: the SMALL capacity for spheres, with planes boxing the camera in on every side."""
    world = World()
    mats = [_diffuse((0.7, 0.3, 0.3)), _diffuse((0.3, 0.7, 0.3), emit=(0.5, 0.5, 0.2)),
            Material(SpecularBRDF(UniformPigment(Color(0.5, 0.5, 0.5))), UniformPigment(Color(0, 0, 0))), _checkered()]
    for i in range(8):
        t = translation(Vec(2.0 * (i % 4) - 2.0, 2.5 * (i // 4) - 1.2, 0.6 + 0.3 * (i % 3))) * scaling(Vec(0.5, 0.5, 0.5))
        world.add_shape(Sphere(t, mats[i % 4]))
    sky = Material(DiffuseBRDF(UniformPigment(Color(0, 0, 0))), UniformPigment(Color(0.7, 0.5, 1)))
    world.add_shape(Plane(Transformation(), mats[3]))
    world.add_shape(Plane(translation(Vec(0, 0, 30)) * rotation_y(10), sky))
    for k, (ax, ang, d) in enumerate([(rotation_x, 90, 12), (rotation_x, -90, 12), (rotation_y, 90, 14), (rotation_y, -90, 14),
                                      (rotation_x, 80, -12), (rotation_y, 85, -14)]):
        world.add_shape(Plane(ax(ang) * translation(Vec(0, 0, d)), mats[k % 3]))
    return world


def _textured():
    """uv-dependent pigments on a sphere: checkered BRDF, image emission; a plane with an image BRDF."""
    tex = scenes.gradient_texture(16, 8)
    world = World()
    world.add_shape(Sphere(translation(Vec(0, 0, 1)) * rotation_z(30),
                           Material(DiffuseBRDF(CheckeredPigment(Color(0.9, 0.2, 0.2), Color(0.2, 0.2, 0.9), 6)), ImagePigment(tex))))
    world.add_shape(Plane(Transformation(), Material(DiffuseBRDF(ImagePigment(tex)), UniformPigment(Color(0, 0, 0)))))
    return world


def _emissive():
    world = World()
    world.add_shape(Sphere(translation(Vec(0, 0, 2)), _diffuse((0.2, 0.2, 0.2), emit=(4.0, 3.5, 3.0))))
    world.add_shape(Sphere(translation(Vec(0, -1.5, 0.8)) * scaling(Vec(0.7, 0.7, 0.7)), _diffuse((0.8, 0.8, 0.8))))
    world.add_shape(Plane(Transformation(), _checkered()))
    return world


SCENES = {"one_plane": _one_plane, "demo": None, "two_spheres": _two_spheres, "largest": _largest, "textured": _textured,
          "emissive": _emissive}
# name: (samples_per_side, path-tracer parameters, error map)
SETTINGS = {
    "spp64": (8, dict(num_of_rays=4, max_depth=5, rr_limit=2), False),
    "spp16": (4, dict(num_of_rays=4, max_depth=5, rr_limit=2), False),
    "n1": (8, dict(num_of_rays=1, max_depth=5, rr_limit=2), False),
    "err": (8, dict(num_of_rays=4, max_depth=5, rr_limit=2), True),
}

_scenes = {}


def scene(name):
    if name not in _scenes:
        if name == "demo":
            flat, cam = demo_flat()
        else:
            flat, cam = flatten_world(SCENES[name]()), flatten_camera(_camera())
        assert flat.n_shapes <= 16
        _scenes[name] = (DeviceScene(flat), cam)
    return _scenes[name]


def render(name, setting):
    """What the fixture pins: {"rgb", "rays"} (per-pixel ray counts) or, for the error map, {"mean", "err"}; and
    the frame's ray count."""
    sc, cam = scene(name)
    S, kw, err = SETTINGS[setting]
    mk = lambda **extra: make_params(W, H, cam, algorithm="pathtracing", samples_per_side=S, background=BG,
                                     aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw, **extra)
    if err:
        mean, e, _, st = sc.render_adaptive(mk(), 0.0, 1)
        out = {"mean": mean, "err": e}
    else:
        rgb, rays, st = sc.render(mk(hit_mode=_abi.RT_HIT_RAY_COUNT), want_hit=True)
        out = {"rgb": rgb, "rays": rays}
    assert st["overflow"] == 0
    out["rays_closest"] = np.array([st["rays_closest"]], dtype=np.int64)
    return out


def fixture_path(name):
    return os.path.join(GOLDEN, f"small_{name}.npz")


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SETTINGS))
@pytest.mark.parametrize("name", list(SCENES))
def test_small_scene_is_pinned(name, setting):
    want = np.load(fixture_path(name))
    got = render(name, setting)
    for key, value in got.items():
        ref = want[f"{setting}_{key}"]
        assert value.dtype == ref.dtype and np.array_equal(value, ref), (key, int((value != ref).sum()))
