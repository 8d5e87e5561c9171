"""Furnaces and their closed forms, in fp64.

A furnace is a closed convex emitter (a sphere or an ellipsoid) with the camera inside it: every ray that starts
inside it or on its inner surface next hits the furnace itself, whatever the BRDF draws and whatever other shapes
lie strictly outside it.  With a uniform albedo rho and emission E per channel, PathTracer.__call__
(render.py:99-139, oracle/pt_oracle.c pathtracer_call) then has answers that hold for any random numbers:

* no roulette (rr_limit > max_depth D): every sample is V = E sum_{d=0..D} rho^d, exactly, and costs
  sum_{d=0..D} N^d closest-hit rays (children at depth D + 1 come back black before they intersect anything);
* rho = 0: `lum > 0` fails, no child is traced: every sample is E and costs one ray;
* N = 1 with roulette from depth R: q = max(0.05, 1 - max_c rho_c), s = 1 / (1 - q), w_j = s for j >= R, else 1.
  A sample that traced k + 1 rays is exactly V(k) = sum_{d=0..k} E prod_{j<d} rho w_j (at k = D killed and
  survived give the same value), and P(k) = 0 for k < R, (1-q)^(k-R) q for R <= k < D, (1-q)^(D-R) at k = D;
* any N with roulette: E[sample] = E sum_{d<=D} rho^d (the roulette is unbiased) and
  E[rays per sample] = sum_{d=0..D} N^d (1-q)^max(0, d-R).

One child escapes all this: a diffuse child whose cos^2(theta) draw is exactly 1 leaves along the tangent plane
(its chord is below tmin) and misses the furnace.  The reference draws it with probability 2^-32 per diffuse bounce.

The `oracle_*` functions evaluate the same recursion in the fp64 operation order of pt_oracle.c, so that the
oracle can be pinned to them bit for bit (tests/test_furnace_cpu.py); the closed forms agree with them to a few
ulps.
"""
from __future__ import annotations

import numpy as np

from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.scene import (
    CheckeredPigment, Color, DiffuseBRDF, ImagePigment, Material, PerspectiveCamera, Plane, SpecularBRDF, Sphere,
    Transformation, UniformPigment, Vec, World, rotation_x, rotation_y, rotation_z, scaling, translation,
)

# --------------------------------------------------------------------------------------------- closed forms


def rays_per_sample(N: int, D: int, rho=None) -> int:
    """Closest-hit rays of one sample without roulette (exact integer)."""
    if D < 0:
        return 0
    if rho is not None and max(rho) <= 0.0:
        return 1
    return sum(N ** d for d in range(D + 1))


def value(E, rho, D: int, d0: int = 0) -> np.ndarray:
    """E sum_{d=d0..D} rho^(d - d0): a ray of depth d0 from inside (d0 = 0: a camera sample), no roulette."""
    E, rho = np.asarray(E, np.float64), np.asarray(rho, np.float64)
    if D < d0:
        return np.zeros(3)
    return E * sum(rho ** d for d in range(D - d0 + 1))


def roulette_q(rho) -> float:
    return max(0.05, 1.0 - float(max(rho)))


def values_by_k(E, rho, R: int, D: int) -> np.ndarray:
    """[D + 1][3]: V(k), the value of an N = 1 sample that traced k + 1 rays, roulette from depth R."""
    E, rho = np.asarray(E, np.float64), np.asarray(rho, np.float64)
    s = 1.0 / (1.0 - roulette_q(rho))
    out, term, acc = np.zeros((D + 1, 3)), np.ones(3), np.zeros(3)
    for k in range(D + 1):
        acc = acc + E * term
        out[k] = acc
        term = term * rho * (s if k >= R else 1.0)
    return out


def law_of_k(rho, R: int, D: int) -> np.ndarray:
    """[D + 1]: P(an N = 1 sample traces k + 1 rays), roulette from depth R."""
    q = roulette_q(rho)
    p = np.zeros(D + 1)
    if R >= D:
        p[D] = 1.0
        return p
    for k in range(R, D):
        p[k] = (1.0 - q) ** (k - R) * q
    p[D] = (1.0 - q) ** (D - R)
    return p


def mean_rays(N: int, rho, R: int, D: int) -> float:
    """E[closest-hit rays per sample] with roulette from depth R."""
    q = roulette_q(rho)
    return float(sum(N ** d * (1.0 - q) ** max(0, d - R) for d in range(D + 1)))


# ------------------------------------------------------------------- the same recursion in pt_oracle.c's order


def _oracle_level(E, hc, v, N):
    out = []
    for c in range(3):
        cum = 0.0
        for _ in range(N):
            cum = cum + hc[c] * v[c]
        out.append(E[c] + cum * (1.0 / N))
    return out


def oracle_value(E, rho, N: int, D: int, d0: int = 0) -> np.ndarray:
    """pathtracer_call's result for a ray of depth d0 from inside, no roulette, in its fp64 operation order."""
    E, rho = [float(x) for x in E], [float(x) for x in rho]
    if D < d0:
        return np.zeros(3)
    v = list(E)  # depth D: the children are cut, cum = 0
    if max(rho) > 0.0:
        for _ in range(D - d0):
            v = _oracle_level(E, rho, v, N)
    return np.array(v)


def oracle_values_by_k(E, rho, R: int, D: int) -> np.ndarray:
    """[D + 1][3]: V(k) for N = 1 with roulette from depth R, in pt_oracle.c's operation order."""
    E, rho = [float(x) for x in E], [float(x) for x in rho]
    lum = max(rho)
    q = max(0.05, 1 - lum)
    kk = 1.0 / (1.0 - q)
    out = np.zeros((D + 1, 3))
    for k in range(D + 1):
        v = list(E)
        for d in range(k - 1, -1, -1):
            hc = [x * kk for x in rho] if d >= R else rho
            v = _oracle_level(E, hc, v, 1)
        out[k] = v
    return out


def oracle_pixel(v, S: int) -> np.ndarray:
    """fire_all_rays' pixel of S^2 equal samples v (imagetracer.py:99-101 order)."""
    if S <= 0:
        return np.asarray(v, np.float64)
    cum = [0.0, 0.0, 0.0]
    for _ in range(S * S):
        cum = [cum[c] + float(v[c]) for c in range(3)]
    w = 1.0 / float(S * S)
    return np.array([x * w for x in cum])


# ------------------------------------------------------------------------------------------------- furnaces

RADIUS = 100.0  # a large furnace: a diffuse child from the inner surface misses it (chord <= tmin = 1e-3)
#                 with probability ~ (5e-4 / radius)^2, below the 2^-32 of the generator's own end point
ELLIPSOID_AXES = (300.0, 150.0, 70.0)
ELLIPSOID_CENTRE = (40.0, -25.0, 12.0)


def _c(x) -> Color:
    return Color(*[float(v) for v in x])


def constant_texture(color, w: int = 5, h: int = 3) -> HdrImage:
    rgb = np.empty((h, w, 3), np.float32)
    rgb[...] = np.asarray(color, np.float32)
    return HdrImage.from_array(rgb)


def furnace_material(rho, E, specular=False, pigments="uniform") -> Material:
    """pigments: "uniform"; "checkered" (BRDF: a CheckeredPigment of two equal colours, emission: an ImagePigment
    of a constant texture); "image" (the other way round)."""
    if pigments == "uniform":
        brdf_p, emit_p = UniformPigment(_c(rho)), UniformPigment(_c(E))
    elif pigments == "checkered":
        brdf_p, emit_p = CheckeredPigment(_c(rho), _c(rho), 3), ImagePigment(constant_texture(E))
    elif pigments == "image":
        brdf_p, emit_p = ImagePigment(constant_texture(rho)), CheckeredPigment(_c(E), _c(E), 4)
    else:
        raise ValueError(pigments)
    brdf = SpecularBRDF(brdf_p) if specular else DiffuseBRDF(brdf_p)
    return Material(brdf, emit_p)


def exact_colors(rho, E, pigments="uniform"):
    """The albedo and emission the flattened scene holds: texels are stored in fp32."""
    rho, E = np.asarray(rho, np.float64), np.asarray(E, np.float64)
    if pigments == "checkered":
        E = E.astype(np.float32).astype(np.float64)
    elif pigments == "image":
        rho = rho.astype(np.float32).astype(np.float64)
    return rho, E


def furnace_shape(kind: str, material: Material):
    """kind: "sphere" (radius RADIUS at the origin) or "ellipsoid" (ELLIPSOID_AXES, rotated, translated)."""
    if kind == "sphere":
        return Sphere(scaling(Vec(RADIUS, RADIUS, RADIUS)), material)
    t = (translation(Vec(*ELLIPSOID_CENTRE)) * rotation_z(27.0) * rotation_y(-41.0) * rotation_x(13.0)
         * scaling(Vec(*ELLIPSOID_AXES)))
    return Sphere(t, material)


def furnace_camera(kind: str) -> PerspectiveCamera:
    """Inside the furnace, off its centre, looking along a tilted axis."""
    ofs = (30.0, -20.0, 10.0) if kind == "sphere" else tuple(c + d for c, d in zip(ELLIPSOID_CENTRE, (25.0, 15.0, -10.0)))
    t = translation(Vec(*ofs)) * rotation_z(35.0) * rotation_y(-20.0)
    return PerspectiveCamera(screen_distance=1.0, aspect_ratio=47 / 29, transformation=t)


def decoys(n_spheres: int, n_planes: int, kind: str, seed: int = 7):
    """Spheres and planes strictly outside the furnace, bright and emitting, so that a ray reaching one of them
    changes the answer.  Spheres: centres 2.5 to 8 bounding radii away,
    radii at most a third of a bounding radius; planes: 1.5 to 3 bounding radii from the centre."""
    rng = np.random.default_rng(seed)
    centre = np.zeros(3) if kind == "sphere" else np.array(ELLIPSOID_CENTRE)
    bound = RADIUS if kind == "sphere" else max(ELLIPSOID_AXES)
    mat = Material(DiffuseBRDF(UniformPigment(Color(0.9, 0.9, 0.9))), UniformPigment(Color(7.0, 11.0, 13.0)))
    spheres = []
    for _ in range(n_spheres):
        d = rng.normal(size=3)
        d /= np.linalg.norm(d)
        c = centre + d * bound * rng.uniform(2.5, 8.0)
        r = bound * rng.uniform(0.05, 0.33)
        spheres.append(Sphere(translation(Vec(*c)) * scaling(Vec(r, r, r)), mat))
    planes = []
    for i in range(n_planes):
        # a plane z = 0 rotated about x and y, pushed out along its own normal
        dist = bound * rng.uniform(1.5, 3.0)
        t = (translation(Vec(*centre)) * rotation_x(float(rng.uniform(0, 360))) * rotation_y(float(rng.uniform(0, 360)))
             * translation(Vec(0.0, 0.0, dist if i % 2 == 0 else -dist)))
        planes.append(Plane(t, mat))
    return spheres, planes


def furnace_world(kind: str, material: Material, n_spheres: int = 0, n_planes: int = 0):
    """World with the decoys first (planes interleaved between the spheres) and the furnace last: the index a
    kernel reports for the furnace has to be mapped back to World order.  Returns (world, furnace index)."""
    spheres, planes = decoys(n_spheres, n_planes, kind)
    world = World()
    order = []
    while spheres or planes:
        if spheres:
            order.append(spheres.pop())
        if planes:
            order.append(planes.pop())
    for s in order:
        world.add_shape(s)
    world.add_shape(furnace_shape(kind, material))
    return world, len(world.shapes) - 1


def chi2_pvalue(ks: np.ndarray, law: np.ndarray) -> float:
    """Pearson chi-square p-value of the observed k (one per sample) against `law`, adjacent bins merged from
    the right until each expects at least 5 samples; impossible k (law 0) observed gives p = 0."""
    from scipy import stats

    ks = np.asarray(ks)
    n = ks.size
    obs = np.bincount(ks, minlength=law.size).astype(np.float64)
    if obs.size > law.size or (obs[law == 0] > 0).any():
        return 0.0
    keep = law > 0
    obs, exp = obs[keep], law[keep] * n
    o_bins, e_bins, o_acc, e_acc = [], [], 0.0, 0.0
    for o, e in zip(obs[::-1], exp[::-1]):
        o_acc, e_acc = o_acc + o, e_acc + e
        if e_acc >= 5.0:
            o_bins.append(o_acc)
            e_bins.append(e_acc)
            o_acc = e_acc = 0.0
    if e_acc > 0 and e_bins:
        o_bins[-1] += o_acc
        e_bins[-1] += e_acc
    if len(e_bins) < 2:
        return 1.0
    return float(stats.chisquare(o_bins, e_bins).pvalue)


# name: (shape, specular BRDF, pigments, rho, E); every rho and E differs per channel, so that a mixed-up channel
# shows; max rho 0.8 (q = 0.2), 0.97 (q at the 0.05 floor) and 0 (no child is ever traced)
FURNACES = {
    "diffuse": ("sphere", False, "uniform", (0.8, 0.55, 0.3), (0.9, 0.35, 0.6)),
    "mirror": ("sphere", True, "uniform", (0.6, 0.97, 0.25), (0.2, 0.7, 0.45)),
    "ellipsoid": ("ellipsoid", False, "uniform", (0.35, 0.5, 0.97), (0.5, 0.8, 0.3)),
    "checkered": ("sphere", False, "checkered", (0.8, 0.3, 0.55), (0.45, 0.9, 0.25)),
    "image": ("ellipsoid", True, "image", (0.97, 0.4, 0.7), (0.3, 0.6, 0.95)),
    "black": ("sphere", False, "uniform", (0.0, 0.0, 0.0), (0.7, 0.2, 0.4)),
}


def furnace(name: str, n_spheres: int = 0, n_planes: int = 0):
    """(world, furnace index in World order, camera, rho, E) with rho and E as the flattened scene holds them."""
    kind, specular, pigments, rho, E = FURNACES[name]
    world, idx = furnace_world(kind, furnace_material(rho, E, specular, pigments), n_spheres, n_planes)
    rho, E = exact_colors(rho, E, pigments)
    return world, idx, furnace_camera(kind), rho, E


def inside_rays(name: str, n: int, seed: int = 3) -> np.ndarray:
    """[n][8] rays from the camera position of furnace `name` in random directions (tmin 1e-5, tmax inf)."""
    kind = FURNACES[name][0]
    cam = furnace_camera(kind)
    o = np.array(cam.transformation.m)[:3, 3]
    d = np.random.default_rng(seed).normal(size=(n, 3))
    rays = np.zeros((n, 8))
    rays[:, :3], rays[:, 3:6], rays[:, 6], rays[:, 7] = o, d, 1e-5, np.inf
    return rays
