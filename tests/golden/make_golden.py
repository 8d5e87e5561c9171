#!/usr/bin/env python
"""Generates the golden fixtures of tests/golden/ by running the UNMODIFIED reference.

    PYTHONDONTWRITEBYTECODE=1 PYTHONPATH=/root/reference/src:/root/repo \
        python tests/golden/make_golden.py [--full]

Everything saved here is an output of the reference's own Python classes (pytracer.*), imported
read-only from /root/reference; nothing of ours computes a number in this script (our flatten only
copies the reference objects' fields into arrays so the scenes can be rebuilt where the reference
tree is absent).  --full adds the 1920x1080 renders of BASELINE config 2 (≈4 min of CPU).

Each scene is parsed/built once per process: Scene.world is a class-level default in the
reference (scene_file.py:363) and would accumulate shapes across parses.
"""
import argparse
import hashlib
import io
import math
import os
import sys
import time

import numpy as np

import pytracer  # noqa: F401  (must resolve to /root/reference/src/pytracer)
from pytracer.camera import OrthogonalCamera, PerspectiveCamera
from pytracer.colors import Color, BLACK, WHITE
from pytracer.geometry import Normal, Point, Vec, Vec2d, create_onb_from_z
from pytracer.hdrimages import HdrImage
from pytracer.imagetracer import ImageTracer
from pytracer.lights import PointLight
from pytracer.materials import (CheckeredPigment, DiffuseBRDF, ImagePigment, Material, SpecularBRDF,
                                UniformPigment)
from pytracer.pcg import PCG
from pytracer.ray import Ray
from pytracer.render import FlatRenderer, OnOffRenderer, PathTracer, PointLightRenderer
from pytracer.scene_file import InputStream, parse_scene
from pytracer.shapes import Plane, Sphere
from pytracer.transformations import (Transformation, rotation_x, rotation_y, rotation_z, scaling,
                                      translation)
from pytracer.world import World

from pytracer_b200.flatten import flatten_camera, flatten_world

assert pytracer.__file__.startswith("/root/reference/"), pytracer.__file__
HERE = os.path.dirname(os.path.abspath(__file__))


class Counting:
    """Wraps World.ray_intersection / is_point_visible with call counters (BASELINE.md §3.3)."""

    def __init__(self, world):
        self.world, self.closest, self.shadow = world, 0, 0
        ri, pv = world.ray_intersection, world.is_point_visible

        def ray_intersection(ray):
            self.closest += 1
            return ri(ray)

        def is_point_visible(point, observer_pos):
            self.shadow += 1
            return pv(point=point, observer_pos=observer_pos)

        world.ray_intersection, world.is_point_visible = ray_intersection, is_point_visible

    def reset(self):
        self.closest = self.shadow = 0


def hit_index_image(world, camera, width, height, samples_per_side=0, pcg=None):
    """Index of the closest shape per pixel, by re-running the loop of world.py:55-64 (argmin t,
    strict '<', first wins) with the reference's own Shape.ray_intersection."""
    tracer = ImageTracer(HdrImage(width, height), camera, samples_per_side, pcg or PCG())
    out = np.full((height, width), -1, dtype=np.int32)
    shapes = world.shapes

    def probe(ray):
        best, best_t = -1, None
        for i, shape in enumerate(shapes):
            h = shape.ray_intersection(ray)
            if h and (best_t is None or h.t < best_t):
                best, best_t = i, h.t
        probe.last = best
        return BLACK

    for row in range(height):
        for col in range(width):
            if samples_per_side > 0:
                for ir in range(samples_per_side):
                    for ic in range(samples_per_side):
                        up = (ic + tracer.pcg.random_float()) / samples_per_side
                        vp = (ir + tracer.pcg.random_float()) / samples_per_side
                        probe(tracer.fire_ray(col, row, up, vp))
            else:
                probe(tracer.fire_ray(col, row))
            out[row, col] = probe.last
    return out


def image_array(image):
    return np.array([(p.r, p.g, p.b) for p in image.pixels], dtype=np.float64).reshape(image.height, image.width, 3)


def render(world, camera, width, height, algorithm, samples_per_side, counter, aa_seed=(42, 54),
           pt_seed=(45, 54), **kw):
    image = HdrImage(width, height)
    aa = PCG(*aa_seed)
    tracer = ImageTracer(image, camera, samples_per_side, aa)
    pt = PCG(*pt_seed)
    if algorithm == "onoff":
        renderer = OnOffRenderer(world=world, background_color=kw.get("background", BLACK), color=kw.get("color", WHITE))
    elif algorithm == "flat":
        renderer = FlatRenderer(world=world, background_color=kw.get("background", BLACK))
    elif algorithm == "pointlight":
        renderer = PointLightRenderer(world=world, background_color=kw.get("background", BLACK),
                                      ambient_color=kw.get("ambient", Color(0.1, 0.1, 0.1)))
    else:
        renderer = PathTracer(world=world, background_color=kw.get("background", BLACK), pcg=pt,
                              num_of_rays=kw["num_of_rays"], max_depth=kw["max_depth"],
                              russian_roulette_limit=kw.get("rr_limit", 3))
    counter.reset()
    t0 = time.time()
    tracer.fire_all_rays(renderer)
    dt = time.time() - t0
    return dict(rgb=image_array(image), rays_closest=counter.closest, rays_shadow=counter.shadow,
                aa_state_end=np.uint64(aa.state), pt_state_end=np.uint64(pt.state), seconds=dt)


def second_scene():
    """A scene that exercises what demo.txt does not: image pigment, non-uniformly scaled and
    rotated spheres, a reflection (negative scale), an orthogonal camera, two lights (one with
    linear_radius 0), a diffuse emitter, a specular material lit by point lights."""
    tex = HdrImage(4, 3)
    for y in range(3):
        for x in range(4):
            tex.set_pixel(x, y, Color(0.1 + 0.2 * x, 0.9 - 0.25 * y, 0.3 + 0.05 * x * y))
    m_img = Material(DiffuseBRDF(ImagePigment(tex)), UniformPigment(Color(0.0, 0.0, 0.0)))
    m_chk = Material(DiffuseBRDF(CheckeredPigment(Color(0.9, 0.8, 0.2), Color(0.2, 0.3, 0.9), 6)), UniformPigment(BLACK))
    m_spec = Material(SpecularBRDF(UniformPigment(Color(0.7, 0.7, 0.6))), UniformPigment(BLACK))
    m_emit = Material(DiffuseBRDF(UniformPigment(Color(0.4, 0.4, 0.4))), UniformPigment(Color(0.9, 0.6, 0.3)))
    m_sky = Material(DiffuseBRDF(UniformPigment(BLACK)), CheckeredPigment(Color(0.6, 0.7, 1.0), Color(0.9, 0.9, 0.9), 2))
    w = World()
    w.add_shape(Sphere(translation(Vec(0.3, -0.9, 0.6)) * rotation_z(25.0) * rotation_x(40.0) * scaling(Vec(0.6, 0.9, 0.4)), m_img))
    w.add_shape(Sphere(translation(Vec(0.0, 0.8, 0.5)) * scaling(Vec(0.5, 0.5, 0.5)), m_spec))
    w.add_shape(Sphere(translation(Vec(-0.8, 0.1, 0.35)) * scaling(Vec(0.35, -0.35, 0.35)), m_emit))
    w.add_shape(Sphere(translation(Vec(1.2, 0.2, 1.6)) * rotation_y(70.0) * scaling(Vec(0.3, 0.7, 0.3)), m_chk))
    w.add_shape(Plane(Transformation(), m_chk))
    w.add_shape(Plane(translation(Vec(0.0, 0.0, 30.0)) * rotation_x(10.0), m_sky))
    w.add_light(PointLight(Point(-3.0, 4.0, 6.0), Color(1.0, 0.9, 0.8), 0.0))
    w.add_light(PointLight(Point(2.0, -5.0, 3.0), Color(0.3, 0.4, 0.9), 2.5))
    cam_p = PerspectiveCamera(screen_distance=1.3, aspect_ratio=1.5,
                              transformation=rotation_z(-20.0) * translation(Vec(-3.5, 0.2, 1.1)) * rotation_y(8.0))
    cam_o = OrthogonalCamera(aspect_ratio=1.5, transformation=translation(Vec(-3.0, 0.0, 1.2)) * scaling(Vec(1.0, 1.6, 1.6)))
    return w, cam_p, cam_o


def save(name, **arrays):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrays)
    print(f"wrote {name}: {os.path.getsize(path) / 1024:.1f} KiB")


def flat_dict(prefix, world, camera=None):
    d = {f"{prefix}{k}": v for k, v in flatten_world(world).to_npz_dict().items()}
    if camera is not None:
        cam = flatten_camera(camera)
        d[f"{prefix}camera"] = np.array([cam.kind, cam.screen_distance, cam.aspect_ratio] + list(cam.m), dtype=np.float64)
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true")
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    only = set(args.only.split(",")) if args.only else None

    def want(tag):
        return only is None or tag in only

    with open("/root/reference/examples/demo.txt", "rt") as f:
        scene = parse_scene(InputStream(stream=f, file_name="demo.txt"), variables={})
    demo_world, demo_camera = scene.world, scene.camera
    demo_counter = Counting(demo_world)

    if want("scene"):
        save("demo_scene.npz", **flat_dict("", demo_world, demo_camera))

    # ---- BASELINE config 1: the reference CLI defaults at 160x120, 1 spp
    if want("c1"):
        r = render(demo_world, demo_camera, 160, 120, "pathtracing", 1, demo_counter, num_of_rays=10, max_depth=3)
        print(f"C1: {r['rays_closest']} rays in {r['seconds']:.1f} s, mean {r['rgb'].reshape(-1, 3).mean(0)}")
        save("demo_c1_pathtracing_160x120.npz", **r)

    # ---- deterministic renderers, centre rays and replayed jitter
    if want("det"):
        out = {}
        for algo in ("onoff", "flat", "pointlight"):
            r = render(demo_world, demo_camera, 160, 120, algo, 0, demo_counter)
            for k, v in r.items():
                out[f"{algo}_s0_{k}"] = v
            r = render(demo_world, demo_camera, 64, 48, algo, 2, demo_counter)
            for k, v in r.items():
                out[f"{algo}_s2_{k}"] = v
        out["hit_s0"] = hit_index_image(demo_world, demo_camera, 160, 120, 0)
        out["hit_s2"] = hit_index_image(demo_world, demo_camera, 64, 48, 2, PCG(42, 54))
        save("demo_deterministic.npz", **out)

    # ---- path tracing with roulette inside the tree (rr_limit < max_depth) and N != 10
    if want("pt_small"):
        r = render(demo_world, demo_camera, 40, 30, "pathtracing", 2, demo_counter, num_of_rays=3,
                   max_depth=5, rr_limit=2, aa_seed=(7, 11), pt_seed=(99, 3),
                   background=Color(0.05, 0.02, 0.01))
        print(f"pt_small: {r['rays_closest']} rays in {r['seconds']:.1f} s")
        save("demo_pt_small.npz", **r)

    # ---- second scene: textures, ellipsoids, orthogonal camera, two lights
    if want("scene2"):
        w2, cam_p, cam_o = second_scene()
        c2 = Counting(w2)
        out = flat_dict("", w2, cam_p)
        cam = flatten_camera(cam_o)
        out["camera_ortho"] = np.array([cam.kind, cam.screen_distance, cam.aspect_ratio] + list(cam.m), dtype=np.float64)
        for tag, cam_obj in (("persp", cam_p), ("ortho", cam_o)):
            for algo in ("onoff", "flat", "pointlight"):
                r = render(w2, cam_obj, 96, 64, algo, 0, c2, background=Color(0.02, 0.03, 0.04))
                for k, v in r.items():
                    out[f"{tag}_{algo}_{k}"] = v
            out[f"{tag}_hit"] = hit_index_image(w2, cam_obj, 96, 64, 0)
            r = render(w2, cam_obj, 48, 32, "pathtracing", 2, c2, num_of_rays=4, max_depth=4, rr_limit=2,
                       aa_seed=(5, 9), pt_seed=(123, 77), background=Color(0.02, 0.03, 0.04))
            print(f"scene2 {tag} pt: {r['rays_closest']} rays in {r['seconds']:.1f} s")
            for k, v in r.items():
                out[f"{tag}_pt_{k}"] = v
        save("scene2.npz", **out)

        # ---- per-function known answers on scene 2 (random inputs, reference outputs)
        rng = PCG(2718, 28)
        u = lambda lo, hi: lo + (hi - lo) * rng.random_float()
        n = 1500
        rays = np.zeros((n, 8))
        hits = np.zeros((n, 11))  # shape, t, point3, normal3, uv2, found
        for i in range(n):
            o = Point(u(-4, 4), u(-4, 4), u(0.05, 4))
            d = Vec(u(-1, 1), u(-1, 1), u(-1, 0.6))
            ray = Ray(origin=o, dir=d, tmin=1e-5 if i % 3 else 1e-3)
            rays[i] = [o.x, o.y, o.z, d.x, d.y, d.z, ray.tmin, ray.tmax]
            best, best_t = -1, None
            for k, shape in enumerate(w2.shapes):
                h = shape.ray_intersection(ray)
                if h and (best_t is None or h.t < best_t):
                    best, best_t = k, h.t
            c2.reset()
            h = World.ray_intersection(w2, ray)
            if h:
                hits[i] = [best, h.t, h.world_point.x, h.world_point.y, h.world_point.z, h.normal.x, h.normal.y,
                           h.normal.z, h.surface_point.u, h.surface_point.v, 1]
            else:
                hits[i, 0] = -1
        pairs = np.zeros((n, 6))
        vis = np.zeros(n, dtype=np.uint8)
        for i in range(n):
            p, q = Point(u(-4, 4), u(-4, 4), u(0.05, 5)), Point(u(-3, 3), u(-3, 3), u(0.01, 3))
            pairs[i] = [p.x, p.y, p.z, q.x, q.y, q.z]
            vis[i] = World.is_point_visible(w2, point=p, observer_pos=q)
        # scatter_ray for a diffuse and a specular material, one sequential stream each
        scat_in = np.zeros((400, 9))
        scat_out = {}
        for i in range(400):
            nrm = Normal(u(-1, 1), u(-1, 1), u(-1, 1)).normalize()
            scat_in[i] = [u(-1, 1), u(-1, 1), u(-1, 1), u(-2, 2), u(-2, 2), u(0, 2), nrm.x, nrm.y, nrm.z]
        for tag, brdf in (("diffuse", w2.shapes[0].material.brdf), ("specular", w2.shapes[1].material.brdf)):
            pcg = PCG(17, 5)
            res = np.zeros((400, 8))
            for i, row in enumerate(scat_in):
                r = brdf.scatter_ray(pcg=pcg, incoming_dir=Vec(*row[0:3]), interaction_point=Point(*row[3:6]),
                                     normal=Normal(*row[6:9]), depth=1)
                res[i] = [r.origin.x, r.origin.y, r.origin.z, r.dir.x, r.dir.y, r.dir.z, r.tmin, r.tmax]
            scat_out[tag] = res
            scat_out[tag + "_state_end"] = np.uint64(pcg.state)
        onb_in = scat_in[:, 6:9].copy()
        onb_out = np.zeros((400, 9))
        for i, row in enumerate(onb_in):
            e1, e2, e3 = create_onb_from_z(Normal(*row))
            onb_out[i] = [e1.x, e1.y, e1.z, e2.x, e2.y, e2.z, e3.x, e3.y, e3.z]
        uv = np.array([[u(0, 1), u(0, 1)] for _ in range(600)])
        pig = {}
        pigments = [w2.shapes[0].material.brdf.pigment, w2.shapes[3].material.brdf.pigment,
                    w2.shapes[1].material.brdf.pigment, w2.shapes[5].material.emitted_radiance]
        fw = flatten_world(w2)
        for k, p in enumerate(pigments):
            pig[f"pigment{k}"] = np.array([[c.r, c.g, c.b] for c in (p.get_color(Vec2d(a, b)) for a, b in uv)])
        cam_uv = np.array([[u(0, 1), u(0, 1)] for _ in range(200)])
        cam_rays = {}
        for tag, cam_obj in (("persp", cam_p), ("ortho", cam_o)):
            res = np.zeros((200, 8))
            for i, (a, b) in enumerate(cam_uv):
                r = cam_obj.fire_ray(a, b)
                res[i] = [r.origin.x, r.origin.y, r.origin.z, r.dir.x, r.dir.y, r.dir.z, r.tmin, r.tmax]
            cam_rays[tag] = res
        # explicit-ray renderer calls (Renderer.__call__) incl. non-zero depth
        call_rays = rays[:300].copy()
        call = {}
        for algo in ("onoff", "flat", "pointlight", "pathtracing"):
            pcg = PCG(31, 41)
            if algo == "onoff":
                rend = OnOffRenderer(world=w2, background_color=Color(0.02, 0.03, 0.04))
            elif algo == "flat":
                rend = FlatRenderer(world=w2, background_color=Color(0.02, 0.03, 0.04))
            elif algo == "pointlight":
                rend = PointLightRenderer(world=w2, background_color=Color(0.02, 0.03, 0.04))
            else:
                rend = PathTracer(world=w2, background_color=Color(0.02, 0.03, 0.04), pcg=pcg, num_of_rays=2,
                                  max_depth=4, russian_roulette_limit=1)
            res = np.zeros((300, 3))
            for i, row in enumerate(call_rays):
                ray = Ray(origin=Point(*row[0:3]), dir=Vec(*row[3:6]), tmin=row[6], tmax=row[7], depth=(i % 3) if algo == "pathtracing" else 0)
                c = rend(ray)
                res[i] = [c.r, c.g, c.b]
            call[algo] = res
            call[algo + "_state_end"] = np.uint64(pcg.state)
        save("scene2_kat.npz", rays=rays, hits=hits, pairs=pairs, visible=vis, scatter_in=scat_in,
             onb_in=onb_in, onb_out=onb_out, uv=uv, cam_uv=cam_uv, call_rays=call_rays,
             **{f"scatter_{k}": v for k, v in scat_out.items()}, **pig,
             **{f"cam_{k}": v for k, v in cam_rays.items()}, **{f"call_{k}": v for k, v in call.items()})

    # ---- analytic cases of the reference's own tests, evaluated by the reference
    if want("analytic"):
        out = {}
        pcg = PCG()
        furn = []
        for i in range(5):  # tests/test_all.py:1014-1051
            world = World()
            emitted, reflectance = pcg.random_float(), pcg.random_float() * 0.9
            world.add_shape(Sphere(material=Material(brdf=DiffuseBRDF(pigment=UniformPigment(WHITE * reflectance)),
                                                     emitted_radiance=UniformPigment(WHITE * emitted))))
            state0 = pcg.state
            pt = PathTracer(pcg=pcg, num_of_rays=1, world=world, max_depth=100, russian_roulette_limit=101)
            color = pt(Ray(origin=Point(0, 0, 0), dir=Vec(1, 0, 0)))
            furn.append([emitted, reflectance, color.r, color.g, color.b, emitted / (1.0 - reflectance)])
            out[f"furnace_state0_{i}"] = np.uint64(state0)
            out[f"furnace_state1_{i}"] = np.uint64(pcg.state)
        out["furnace"] = np.array(furn)
        save("analytic.npz", **out)

    if args.full and want("full"):
        out = {}
        for algo in ("onoff", "flat", "pointlight"):
            r = render(demo_world, demo_camera, 1920, 1080, algo, 0, demo_counter)
            print(f"1080p {algo}: {r['rays_closest']}+{r['rays_shadow']} rays in {r['seconds']:.1f} s")
            out[f"{algo}_mean"] = r["rgb"].reshape(-1, 3).mean(0)
            out[f"{algo}_rays"] = np.array([r["rays_closest"], r["rays_shadow"]], dtype=np.int64)
            out[f"{algo}_seconds"] = np.float64(r["seconds"])
            if algo == "flat":
                out["flat_rgb_f32"] = r["rgb"].astype(np.float32)
            elif algo == "pointlight":  # 2.3 MB compressed: stored as the digest of its bytes, the tests re-render it with the oracle
                out["pointlight_rgb_f32_sha256"] = np.str_(hashlib.sha256(r["rgb"].astype(np.float32).tobytes()).hexdigest())
        out["hit"] = hit_index_image(demo_world, demo_camera, 1920, 1080, 0).astype(np.int8)
        save("demo_1080p.npz", **out)


if __name__ == "__main__":
    main()
