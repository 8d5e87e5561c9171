"""Every path-tracer kernel against the closed-form furnace radiance of tests/furnace_ref.py (pinned to the fp64
oracle by tests/test_furnace_cpu.py): k_pt_warp with the scene tables in the SMALL, shared or global form and each
accumulator (ACC_REG, ACC_LANES, ACC_SEG), with and without the error map (ERR); k_pt_warp_bvh; the fp32 and fp64
mega kernels; rt_render_adaptive, the RT_PART_SPP / RT_PART_ROWS shares, rt_trace_rays and rt_render_multi.

Decoy spheres and planes lie strictly outside the furnace, before it in World order: they pick the instantiation
(and make the kernel map the furnace's index back to World order) without changing the answer.

What is checked:
* integers exactly: the per-pixel ray counts (RT_HIT_RAY_COUNT), the hit index (RT_HIT_SHAPE), rays_closest,
  samples, overflow == 0 (an overflowing run fails with RT_ERR_OVERFLOW, which fails the test);
* fp64 values within 1e-12 relative;
* fp32 values within the bound of `fp32_bound` (derived there), the worst deviation printed in units of 2^-24 V;
* the roulette: every N = 1 sample equals V(k) at the k its ray count gives, the histogram of k follows the law of k
  (fixed seeds: the chi-square p-value is deterministic; p >= 1e-6), and for N > 1 the mean value and the mean
  ray count are within 5 sigma of the closed forms.

TANGENT: the furnace is closed for every child but one whose cos^2(theta) draw is exactly 1: it leaves along the
tangent plane and escapes (and may reach a decoy).  The fp64 kernels, like the reference, draw it with probability
2^-32; the fp32 kernels compute the draw as fl(x) * 2^-32, which rounds the 128 largest x to 1, so with probability
2^-25 per diffuse bounce.  Case sizes keep the diffuse bounces of every fp32 render checked sample by sample or pixel by pixel to about
10^6 or fewer (an
expectation of 0.03 such children; with fixed seeds the outcome is deterministic).

Instantiation names in the case ids (tables-accumulator-G, G the pixels of a task) follow the launchers' sizing
rules (launch_pt_warp_impl in rt_warp.cuh, launch_pt_warp_bvh in rt_warp_bvh.cuh), restated in `instantiation`."""
import numpy as np
import pytest

import furnace_ref as fr
from pytracer_b200 import _abi, _native
from pytracer_b200.device import DeviceScene, MultiDeviceScene
from pytracer_b200.flatten import flatten_world
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
NO_RR = 10 ** 6  # rr_limit beyond any depth: no roulette

# decoy set: (spheres, planes, accel).  With the furnace: 5 spheres and 8 shapes (odd plane count) and 8 spheres and
# 16 shapes (even) fit the SMALL tables; 37 spheres' tables (1.9 KB) are staged in shared memory; 1 400 spheres'
# (67 KB) stay in global memory; "bvh" walks the sphere hierarchy (k_pt_warp_bvh, the BVH mega kernels).
DECOYS = {
    "small-odd": (4, 3, "none"),
    "small-even": (7, 8, "none"),
    "smem37": (37, 2, "none"),
    "global1400": (1400, 1, "none"),
    "bvh37": (37, 2, "bvh"),
    "bvh1400": (1400, 1, "bvh"),
}
KERNELS = {
    "warp": dict(variant="warp"),
    "mega32": dict(variant="mega", precision="f32"),
    "mega64": dict(variant="mega", precision="f64", out_f64=True),
}
VARIANT_USED = {"warp": _abi.RT_VARIANT_WARP, "mega32": _abi.RT_VARIANT_MEGA, "mega64": _abi.RT_VARIANT_MEGA}


def instantiation(decoy: str, kernel: str, L: int, N: int, D: int) -> str:
    """The kernel instantiation a render of L samples per pixel reaches (launch_pt_warp_impl: G = 1 for L >= 32,
    else ceil(32 / L) up to 8 for L >= 4, else 32 / L, and at most 32 / L outside the SMALL tables; ACC_REG for
    G = 1, ACC_LANES up to 8, else ACC_SEG, and ACC_SEG also where the ACC_LANES columns cost a resident block;
    launch_pt_warp_bvh: ceil(32 / L) up to 8, accumulator columns)."""
    if kernel != "warp":
        return kernel
    ns, npl, accel = DECOYS[decoy]
    if accel == "bvh":
        return f"bvh-G{min(-(-32 // L), 8)}"
    n_sph, n_sh = ns + 1, ns + npl + 1
    small = n_sph <= 8 and n_sh <= 16
    shape_bytes = (n_sph + 1) // 2 * 96 + npl * 48
    tables = "small" if small else ("smem" if shape_bytes <= 64 * 1024 else "global")
    G = 1 if L >= 32 else (min(-(-32 // L), 8) if L >= 4 else 32 // L)
    if G * L > 32 and not small:
        G = max(32 // L, 1)
    acc = "REG" if G == 1 else ("LANES" if G <= 8 else "SEG")
    if acc == "LANES":
        cap = max(-(-G * L // 32) * 32 + (32 if N == 1 else 32 * D), 64)
        shape = 3648 if small else (-(-shape_bytes // 16) * 16 if tables == "smem" else 0)
        rec = (cap + 1) * 48 + 32 * 4
        blocks = lambda pw: min((227 * 1024) // (shape + 8 * pw + 1024), 8, 3 if small else 2)
        if blocks(rec + 96 * 4) > blocks(rec + G * 96 * 4):
            acc = "SEG"
    return f"{tables}-{acc}-G{G}"


def fp32_bound(D: int, n_terms: int, roulette_levels: int = 0) -> float:
    """Relative error bound of an fp32 pixel (or sample) value V against the closed form.

    A pixel is the sum of n_terms ray contributions thr_d * E (every ray of every sample hits the furnace), times
    1/S^2.  With u = 2^-24 and every fp32 operation correctly rounded:
    * rho, E and 1/N are fp32 values: 1 rounding each (relative u);
    * thr_{d+1} = (1/N) * (thr_d * rho): 2 products, so with the representations of rho and 1/N 4 roundings per
      depth level, 4 D at most;
    * a roulette survival scales rho by fast_rcp(1 - q) (rcp.approx, within 2u), with q and 1 - q rounded once
      each and one more product: 5 roundings per level of roulette;
    * thr_d * E: E's representation and the product, 2;
    * the sum of n_terms positive terms, in whatever order the accumulator adds them (any binary tree of additions,
      atomics included): at most n_terms - 1 roundings of the total;
    * 1/S^2, its product, and the store to an fp32 image (the mega kernel sums samples in fp64): 3.
    K roundings of at most u each give at most gamma_K = K u / (1 - K u) relative."""
    K = 4 * max(D, 0) + 5 * roulette_levels + 2 + (n_terms - 1) + 3
    return K * U / (1.0 - K * U)


_scenes = {}


def scene(name: str, decoy: str):
    key = (name, decoy)
    if key not in _scenes:
        ns, npl, _ = DECOYS[decoy]
        world, idx, cam, rho, E = fr.furnace(name, ns, npl)
        _scenes[key] = (DeviceScene(flatten_world(world)), idx, cam, rho, E)
    return _scenes[key]


def params(cam, W, H, S, N, D, kernel, accel, R=NO_RR, hit_mode=_abi.RT_HIT_SHAPE, **kw):
    return make_params(W, H, cam, "pathtracing", S, num_of_rays=N, max_depth=D, rr_limit=R, aa_pcg=PCG(42, 54),
                       pt_pcg=PCG(45, 54), accel=accel, hit_mode=hit_mode, **{**KERNELS.get(kernel, {}), **kw})


def deviation(img, V) -> np.ndarray:
    """|img - V| / V per value (V > 0 in every channel)."""
    return np.abs(np.asarray(img, np.float64) - V) / V


def assert_values(img, V, kernel, bound32, what=""):
    """fp64: within 1e-12; fp32: within bound32.  Returns the worst deviation in units of 2^-24 V."""
    dev = deviation(img, V)
    bound = 1e-12 if kernel == "mega64" else bound32
    worst = float(dev.max())
    assert worst <= bound, f"{what}: worst relative deviation {worst:.3e} = {worst / U:.1f} u > {bound / U:.1f} u"
    return worst / U


WORST = {}  # kernel -> worst fp32 deviation seen, in units of 2^-24 V (printed at the end of the module)


def _note(kernel, instance, ulps):
    key = kernel if kernel != "warp" else f"warp {instance}"
    WORST[key] = max(WORST.get(key, 0.0), ulps)


def exact_case(name, decoy, kernel, W, H, S, N, D):
    sc, idx, cam, rho, E = scene(name, decoy)
    accel = DECOYS[decoy][2]
    spp = max(S, 1) ** 2
    R1 = fr.rays_per_sample(N, D, rho)
    V = fr.value(E, rho, D)
    inst = instantiation(decoy, kernel, spp, N, D)
    rgb, hit, st = sc.render(params(cam, W, H, S, N, D, kernel, accel), want_hit=True)
    rgb2, rays, st2 = sc.render(params(cam, W, H, S, N, D, kernel, accel, hit_mode=_abi.RT_HIT_RAY_COUNT), want_hit=True)
    for s in (st, st2):
        assert s["overflow"] == 0 and s["variant_used"] == VARIANT_USED[kernel]
        assert s["samples"] == W * H * spp
        assert s["rays_closest"] == W * H * spp * R1, (s["rays_closest"], W * H * spp * R1)
    assert (hit == idx).all(), np.unique(hit)
    assert (rays == spp * R1).all(), np.unique(rays)
    b = fp32_bound(D, spp * R1)
    ulps = max(assert_values(rgb, V, kernel, b, inst), assert_values(rgb2, V, kernel, b, inst))
    _note(kernel, inst, ulps if kernel != "mega64" else 0.0)
    print(f"\n{name}/{decoy}/{kernel} [{inst}] {W}x{H} S = {S} N = {N} D = {D}: {R1} rays per sample, worst "
          f"{ulps:.1f} u (bound {b / U:.0f} u)")


# ------------------------------------------------------------------------------------------------ layouts
LAYOUTS = (
    [("diffuse", d, "warp", 47, 29, S, 2, 3) for d in DECOYS for S in (1, 2, 3, 4, 5, 6, 8)]
    + [("diffuse", d, "warp", w, h, S, 2, 3) for d in ("small-odd", "global1400", "bvh37") for w, h in ((1, 1), (33, 1))
       for S in (1, 3, 8)]
    + [(f, d, "warp", 47, 29, S, 2, 3) for f in ("mirror", "ellipsoid", "checkered", "image", "black")
       for d in ("small-even", "smem37", "bvh1400") for S in (2, 5)]
    + [(f, d, k, 47, 29, 2, 2, 3) for k in ("mega32", "mega64") for f in fr.FURNACES
       for d in ("small-odd", "global1400", "bvh37")]
    + [("ellipsoid", d, k, 33, 1, S, 2, 3) for k in ("mega32", "mega64") for d in ("small-even", "bvh1400") for S in (1, 3)]
)
# (N, D) at the edges of the work stacks: N = 1 chains, N = 40 and N = 1100 (beyond the multiply-shift x / N of the
# warp kernels' record bookkeeping), depth 0, and depth 1022, the deepest the warp record's 10 depth bits hold.
# The edges with thousands of rays per sample run on a 33 x 1 image (partial last tasks still): see TANGENT.
HEAVY = {(40, 2), (1100, 1), (1, 1022)}


def _size(N, D):
    return (33, 1) if (N, D) in HEAVY else (47, 29)


EDGES = [(f, d, k, *_size(N, D), 2, N, D) for N, D in ((1, 8), (2, 6), (40, 2), (1100, 1), (3, 0), (1, 1022))
         for k in KERNELS for f, d in (("diffuse", "small-odd"), ("mirror", "smem37"), ("ellipsoid", "bvh37"))]
EDGES += [("image", "global1400", "warp", *_size(N, D), 2, N, D) for N, D in ((1, 8), (40, 2), (1100, 1), (3, 0))]
EDGES += [("checkered", "bvh1400", "warp", *_size(N, D), 3, N, D) for N, D in ((2, 6), (1100, 1), (1, 1022))]


def _id(c):
    name, decoy, kernel, W, H, S, N, D = c
    return f"{name}-{decoy}-{kernel}[{instantiation(decoy, kernel, max(S, 1) ** 2, N, D)}]-{W}x{H}-S{S}-N{N}-D{D}"


@pytest.mark.parametrize("case", LAYOUTS + EDGES, ids=_id)
def test_furnace_is_exact(case):
    exact_case(*case)


# ------------------------------------------------------------------------------------------- depth limits
def test_depth_1023_selects_mega_and_warp_refuses_it():
    sc, idx, cam, rho, E = scene("diffuse", "small-odd")
    W, H, D = 8, 4, 1023
    rgb, rays, st = sc.render(params(cam, W, H, 1, 1, D, "auto", "none", hit_mode=_abi.RT_HIT_RAY_COUNT), want_hit=True)
    assert st["variant_used"] == _abi.RT_VARIANT_MEGA and st["overflow"] == 0
    assert (rays == D + 1).all() and st["rays_closest"] == W * H * (D + 1)
    assert_values(rgb, fr.value(E, rho, D), "mega32", fp32_bound(D, D + 1))
    with pytest.raises(_native.NativeError) as e:
        sc.render(params(cam, W, H, 1, 1, D, "warp", "none"))
    assert e.value.code == _abi.RT_ERR_INVALID


@pytest.mark.parametrize("kernel", ["warp", "mega32", "mega64", "auto"])
@pytest.mark.parametrize("hit_mode", [_abi.RT_HIT_SHAPE, _abi.RT_HIT_RAY_COUNT], ids=["shape", "ray-count"])
def test_negative_depth_traces_nothing(kernel, hit_mode):
    sc, idx, cam, rho, E = scene("diffuse", "small-odd")
    rgb, hit, st = sc.render(params(cam, 13, 7, 2, 3, -1, kernel, "none", hit_mode=hit_mode), want_hit=True)
    assert (rgb == 0).all() and st["rays_closest"] == 0 and st["samples"] == 13 * 7 * 4 and st["overflow"] == 0
    assert (hit == (0 if hit_mode == _abi.RT_HIT_RAY_COUNT else -1)).all(), np.unique(hit)


# --------------------------------------------------------------------------------------------- roulette
RR1 = ([(f, d, k, D, R) for f, d in (("diffuse", "small-odd"), ("mirror", "smem37"), ("ellipsoid", "bvh37"))
        for k in KERNELS for D, R in ((12, 2), (30, 0))]
       + [("checkered", "global1400", "warp", 12, 2), ("image", "bvh1400", "warp", 30, 0)])
SAMPLES_W, SAMPLES_H = 160, 120  # 19 200 samples, one per pixel at S = 1


def _per_sample_check(rgb, rays, E, rho, R, D, kernel, scale=1.0, what=""):
    """Every sample (pixel * scale) equals V(k), k = its ray count - 1; returns k."""
    k = rays.astype(np.int64) - 1
    assert (k >= min(R, D)).all() and (k <= D).all(), (k.min(), k.max())
    Vk = fr.values_by_k(E, rho, R, D)
    worst = 0.0
    for kk in np.unique(k):
        m = k == kk
        b = fp32_bound(int(kk), int(kk) + 1, max(0, int(kk) - R))
        worst = max(worst, assert_values(np.asarray(rgb, np.float64)[m] * scale, Vk[kk], kernel, b, f"{what} k = {kk}"))
    return k, worst


@pytest.mark.parametrize("case", RR1, ids=lambda c: f"{c[0]}-{c[1]}-{c[2]}[{instantiation(c[1], c[2], 1, 1, c[3])}]-D{c[3]}-R{c[4]}")
def test_roulette_n1_samples_and_law(case):
    name, decoy, kernel, D, R = case
    sc, idx, cam, rho, E = scene(name, decoy)
    accel = DECOYS[decoy][2]
    rgb, rays, st = sc.render(params(cam, SAMPLES_W, SAMPLES_H, 1, 1, D, kernel, accel, R=R, hit_mode=_abi.RT_HIT_RAY_COUNT),
                              want_hit=True)
    assert st["overflow"] == 0 and st["samples"] == SAMPLES_W * SAMPLES_H and st["rays_closest"] == int(rays.sum())
    k, worst = _per_sample_check(rgb, rays, E, rho, R, D, kernel, what=kernel)
    pv = fr.chi2_pvalue(k.ravel(), fr.law_of_k(rho, R, D))
    _note(kernel, instantiation(decoy, kernel, 1, 1, D), worst if kernel != "mega64" else 0.0)
    print(f"\n{name}/{decoy}/{kernel} D = {D} R = {R}: chi-square p = {pv:.4f}, mean k {k.mean():.3f}, worst {worst:.1f} u")
    assert pv >= 1e-6


@pytest.mark.parametrize("decoy", ["small-odd", "smem37", "global1400", "bvh37"])
def test_roulette_n1_spp_partition_samples(decoy):
    """RT_PART_SPP share r of S^2 is sample r of every pixel: the same admissible set, through the partition path."""
    sc, idx, cam, rho, E = scene("diffuse", decoy)
    accel = DECOYS[decoy][2]
    S, D, R = 4, 12, 2
    ks = []
    for r in (0, 5, 15):
        img, rays, st = sc.render(params(cam, 47, 29, S, 1, D, "warp", accel, R=R, hit_mode=_abi.RT_HIT_RAY_COUNT,
                                         part_mode=_abi.RT_PART_SPP, part_count=S * S, part_rank=r), want_hit=True)
        assert st["overflow"] == 0 and st["samples"] == 47 * 29 and st["rays_closest"] == int(rays.sum())
        k, _ = _per_sample_check(img, rays, E, rho, R, D, "warp", scale=S * S, what=f"rank {r}")
        ks.append(k.ravel())
    assert fr.chi2_pvalue(np.concatenate(ks), fr.law_of_k(rho, R, D)) >= 1e-6


RRN = [(f, d, k) for f, d in (("diffuse", "small-odd"), ("mirror", "global1400"), ("ellipsoid", "bvh37")) for k in KERNELS]


@pytest.mark.parametrize("case", RRN, ids=lambda c: "-".join(c))
def test_roulette_many_rays_is_unbiased(case):
    name, decoy, kernel = case
    N, D, R = 3, 5, 2
    sc, idx, cam, rho, E = scene(name, decoy)
    rgb, rays, st = sc.render(params(cam, SAMPLES_W, SAMPLES_H, 1, N, D, kernel, DECOYS[decoy][2], R=R,
                                     hit_mode=_abi.RT_HIT_RAY_COUNT), want_hit=True)
    assert st["overflow"] == 0 and st["rays_closest"] == int(rays.sum())
    x = np.asarray(rgb, np.float64).reshape(-1, 3)
    n = x.shape[0]
    V, mr = fr.value(E, rho, D), fr.mean_rays(N, rho, R, D)
    zv = (x.mean(0) - V) / (x.std(0, ddof=1) / np.sqrt(n))
    zr = (rays.mean() - mr) / (rays.std(ddof=1) / np.sqrt(n))
    print(f"\n{name}/{decoy}/{kernel}: value z {np.round(zv, 2)}, rays z {zr:.2f} (mean {rays.mean():.2f} vs {mr:.2f})")
    assert (np.abs(zv) <= 5).all() and abs(zr) <= 5


# ---------------------------------------------------------------------------------------- entry points
ADAPTIVE = ([("diffuse", d, S) for d in ("small-odd", "smem37", "global1400", "bvh37") for S in (2, 3, 4, 8)]
            + [(f, d, 4) for f in ("mirror", "ellipsoid", "image") for d in ("small-even", "bvh1400")])


@pytest.mark.parametrize("case", ADAPTIVE, ids=lambda c: f"{c[0]}-{c[1]}-S{c[2]}[{instantiation(c[1], 'warp', c[2] ** 2, 2, 3)}-ERR]")
def test_adaptive_zero_variance_is_one_exact_pass(case):
    name, decoy, S = case
    N, D = 2, 3
    sc, idx, cam, rho, E = scene(name, decoy)
    V = fr.value(E, rho, D)
    R1 = fr.rays_per_sample(N, D, rho)
    p = params(cam, 47, 29, S, N, D, "warp", DECOYS[decoy][2])
    mean, err, samples, st = sc.render_adaptive(p, 1e-3, 4, error_floor=1e-2)
    b = fp32_bound(D, S * S * R1)
    assert st["passes"] == 1 and (samples == S * S).all() and st["overflow"] == 0
    assert st["rays_closest"] == 47 * 29 * S * S * R1 and st["samples"] == 47 * 29 * S * S
    ulps = assert_values(mean, V, "warp", b, "adaptive mean")
    # every batch mean is V within b V, so it is within 2 b V of the pixel mean, and a standard error over B >= 2
    # batches, sqrt(sum (x_b - m)^2 / ((B - 1) B)), is at most the largest such distance
    assert (err <= 2 * b * V).all(), float((err / V).max())
    print(f"\n{name}/{decoy} S = {S}: mean worst {ulps:.1f} u, largest err {float((err / V).max()) / U:.1f} u")


@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("decoy", ["small-odd", "global1400", "bvh37"])
def test_partition_shares_sum_to_the_furnace(kernel, decoy):
    sc, idx, cam, rho, E = scene("ellipsoid", decoy)
    accel = DECOYS[decoy][2]
    W, H, S, N, D = 47, 29, 3, 2, 4
    V, R1 = fr.value(E, rho, D), fr.rays_per_sample(N, D, rho)
    for mode, count in ((_abi.RT_PART_SPP, 4), (_abi.RT_PART_ROWS, 3)):
        total = np.zeros((H, W, 3))
        rays_total = np.zeros((H, W), np.int64)
        for r in range(count):
            img, rays, st = sc.render(params(cam, W, H, S, N, D, kernel, accel, hit_mode=_abi.RT_HIT_RAY_COUNT,
                                             part_mode=mode, part_count=count, part_rank=r), want_hit=True)
            assert st["overflow"] == 0 and st["rays_closest"] == int(rays.sum())
            total += img
            rays_total += rays
        assert (rays_total == S * S * R1).all(), np.unique(rays_total)
        assert_values(total, V, kernel, fp32_bound(D, S * S * R1 + count), f"mode {mode}")


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("decoy", ["small-odd", "global1400", "bvh37"])
@pytest.mark.parametrize("d0", [0, 1, 3, 5])
def test_trace_rays_from_inside(precision, decoy, d0):
    name = "diffuse" if decoy != "bvh37" else "ellipsoid"
    sc, idx, cam, rho, E = scene(name, decoy)
    N, D = 2, 5
    rays = fr.inside_rays(name, 64)
    p = params(cam, 1, 1, 0, N, D, "", DECOYS[decoy][2], precision=precision)
    out, _ = sc.trace_rays(p, rays, depth=np.full(64, d0, np.int32))
    V = fr.value(E, rho, D, d0)
    assert_values(out, V, "mega64" if precision == "f64" else "mega32", fp32_bound(D - d0, fr.rays_per_sample(N, D - d0)))


def test_multi_device_furnace():
    n = _native.load().rt_device_count()
    if n < 2:
        pytest.skip("one device visible")
    ns, npl, _ = DECOYS["global1400"]
    world, idx, cam, rho, E = fr.furnace("diffuse", ns, npl)
    multi = MultiDeviceScene(flatten_world(world), min(n, 4))
    W, H, S, N, D = 47, 29, 3, 2, 4
    R1 = fr.rays_per_sample(N, D, rho)
    rgb, rays, st = multi.render(params(cam, W, H, S, N, D, "warp", "none", hit_mode=_abi.RT_HIT_RAY_COUNT), want_hit=True)
    multi.close()
    assert st["overflow"] == 0 and st["rays_closest"] == W * H * S * S * R1 and (rays == S * S * R1).all()
    assert_values(rgb, fr.value(E, rho, D), "warp", fp32_bound(D, S * S * R1))


def test_zz_report_worst_fp32_deviation():
    """(runs last in the module) the worst fp32 deviation per kernel over the cases above, in units of 2^-24 V"""
    print("\nworst fp32 deviation per kernel (units of 2^-24 V): "
          + ", ".join(f"{k} {v:.1f}" for k, v in sorted(WORST.items())))
