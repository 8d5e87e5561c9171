"""Parity of the CUDA path (through the C-ABI) against the oracle and the reference's goldens.

Bars (BASELINE.json north_star): deterministic renderers — hit mask / shape index bit-exact,
colours within 1e-5 relative; path tracing — the reference image itself in replay mode (same
random numbers, fp32 vs fp64 rounding only), and statistical agreement for the parallel streams:
per-pixel means within 3 sigma of the Monte Carlo error and image-mean luminance within 0.5 %.
"""
import numpy as np
import pytest

from oracle import oracle
from pytracer_b200 import _abi, device, scenes
from pytracer_b200.device import DeviceScene
from pytracer_b200.flatten import flatten_camera, flatten_world
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG
from util import assert_luminance_agreement, assert_mc_agreement, c1_params, demo_flat, golden, luminosity, scene2_flat, sha256_of

pytestmark = pytest.mark.gpu

REL = 1e-5  # colour tolerance fp32 vs Python fp64 stated by the north star


def assert_colors_close(got, ref, rel=REL, frac_ok=1.0):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    bad = np.abs(got - ref) > rel * np.maximum(np.abs(ref), 1e-3)
    assert bad.mean() <= 1.0 - frac_ok, f"{bad.sum()} of {bad.size} colour values differ by more than {rel} relative"


# ------------------------------------------------------------------ PCG (tests/test_all.py:872-887)
def test_device_pcg_known_answers():
    state, inc = device.pcg_seed(42, 54)
    assert (state, inc) == (1753877967969059832, 109)
    draws, end = device.pcg_draw(state, inc, 6)
    assert draws.tolist() == [2707161783, 2068313097, 3122475824, 2211639955, 3215226955, 3421331566]
    ref, ref_end = oracle.pcg_draw(state, inc, 1000)
    got, got_end = device.pcg_draw(state, inc, 1000)
    assert np.array_equal(ref, got) and ref_end == got_end


# ------------------------------------------------------------------ per-function known answers
def test_closest_hit_known_answers_fp64_and_fp32():
    fs, _, _ = scene2_flat()
    k = golden("scene2_kat.npz")
    sc = DeviceScene(fs)
    hits64 = sc.intersect(k["rays"], "f64")
    hits32 = sc.intersect(k["rays"], "f32")
    n_mismatch32 = 0
    for h64, h32, ref in zip(hits64, hits32, k["hits"]):
        assert h64.shape == int(ref[0])  # bit-exact index in fp64
        n_mismatch32 += h32.shape != int(ref[0])
        if h64.shape >= 0:
            got = np.array([h64.t, *h64.world_point, *h64.normal, *h64.uv])
            assert np.allclose(got, ref[1:10], rtol=1e-12, atol=1e-12)
            if h32.shape == h64.shape:
                got32 = np.array([h32.t, *h32.world_point, *h32.normal])
                assert np.allclose(got32, ref[1:8], rtol=2e-4, atol=2e-4)
    assert n_mismatch32 <= 2  # grazing rays only
    assert np.array_equal(sc.is_point_visible(k["pairs"], "f64"), k["visible"].astype(bool))
    assert (sc.is_point_visible(k["pairs"], "f32") != k["visible"].astype(bool)).sum() <= 2


def test_scatter_onb_pigments_cameras_known_answers():
    fs, cam_p, cam_o = scene2_flat()
    k = golden("scene2_kat.npz")
    sc = DeviceScene(fs)
    st, inc = 0, 0
    st, inc = oracle.pcg_seed(17, 5)
    for mat, tag in ((0, "diffuse"), (1, "specular")):
        out, end = sc.scatter(mat, k["scatter_in"], st, inc, "f64")
        assert np.allclose(out, k[f"scatter_{tag}"], rtol=1e-12, atol=1e-13)
        assert end == int(k[f"scatter_{tag}_state_end"])
        out32, end32 = sc.scatter(mat, k["scatter_in"], st, inc, "f32")
        assert np.allclose(out32, k[f"scatter_{tag}"], rtol=1e-4, atol=2e-6) and end32 == end
    assert np.allclose(device.onb(k["onb_in"], "f64"), k["onb_out"], rtol=1e-13, atol=1e-15)
    e = device.onb(k["onb_in"], "f32").reshape(-1, 3, 3)  # tests/test_all.py:991-1011: orthonormal
    gram = np.einsum("nij,nkj->nik", e, e)
    assert np.allclose(gram, np.eye(3)[None], atol=1e-5)
    mats = fs.materials
    idx = [mats[fs.shape_material[0]].brdf_pigment, mats[fs.shape_material[3]].brdf_pigment,
           mats[fs.shape_material[1]].brdf_pigment, mats[fs.shape_material[5]].emitted_pigment]
    for j, pig in enumerate(idx):
        assert np.array_equal(sc.pigment_color(pig, k["uv"], "f64"), k[f"pigment{j}"])
        got32 = sc.pigment_color(pig, k["uv"], "f32")  # texture unit / fp32 checker cells
        assert (np.abs(got32 - k[f"pigment{j}"]).max(axis=1) > 1e-6).mean() < 0.01
    for cam, tag in ((cam_p, "persp"), (cam_o, "ortho")):
        assert np.array_equal(device.camera_fire(cam, k["cam_uv"], "f64"), k[f"cam_{tag}"])


def test_image_tracer_rays_replay_the_jitter_stream():
    """imagetracer.py:80-101: sample k uses draws 2k, 2k+1 — the device jumps ahead, the oracle
    draws sequentially; the rays must be identical (tests/test_all.py:556-604 restated)."""
    _, cam_p, cam_o = scene2_flat()
    for cam in (cam_p, cam_o):
        for S in (0, 1, 3):
            p = make_params(37, 23, cam, "flat", S, aa_pcg=PCG(42, 54))
            assert np.array_equal(device.camera_rays(p, "f64"), oracle.camera_rays(p))


def test_renderer_call_on_explicit_rays():
    fs, cam_p, _ = scene2_flat()
    k = golden("scene2_kat.npz")
    sc = DeviceScene(fs)
    bg = (0.02, 0.03, 0.04)
    for algo in ("onoff", "flat", "pointlight"):
        p = make_params(1, 1, cam_p, algo, background=bg, precision="f64")
        out, _ = sc.trace_rays(p, k["call_rays"])
        assert np.allclose(out, k[f"call_{algo}"], rtol=1e-12, atol=1e-14), algo
    pcg = PCG(31, 41)
    p = make_params(1, 1, cam_p, "pathtracing", num_of_rays=2, max_depth=4, rr_limit=1, background=bg, pt_pcg=pcg, precision="f64")
    depth = np.arange(300, dtype=np.int32) % 3
    out, (state, _) = sc.trace_rays(p, k["call_rays"], depth)
    assert state == int(k["call_pathtracing_state_end"])  # same number of draws, same order
    assert np.allclose(out, k["call_pathtracing"], rtol=1e-9, atol=1e-12)


# ------------------------------------------------------------------ deterministic renderers
@pytest.mark.parametrize("algo", ["onoff", "flat", "pointlight"])
@pytest.mark.parametrize("s,size", [(0, (160, 120)), (2, (64, 48))])
def test_demo_deterministic_vs_reference(algo, s, size):
    fs, cam = demo_flat()
    g = golden("demo_deterministic.npz")
    sc = DeviceScene(fs)
    p = make_params(size[0], size[1], cam, algo, s, aa_pcg=PCG(42, 54), out_f64=True)
    rgb, hit, stats = sc.render(p, want_hit=True)
    # AUTO = the hybrid path (fp32 conservative gate + the reference's fp64 decisions); the plain fp64 kernel
    # must give the very same image
    assert stats["precision_used"] == _abi.RT_PRECISION_HYBRID
    assert np.array_equal(hit, g[f"hit_s{s}"])
    assert np.allclose(rgb, g[f"{algo}_s{s}_rgb"], rtol=1e-12, atol=1e-15)
    assert stats["rays_closest"] == int(g[f"{algo}_s{s}_rays_closest"])
    assert stats["rays_shadow"] == int(g[f"{algo}_s{s}_rays_shadow"])
    p64 = make_params(size[0], size[1], cam, algo, s, aa_pcg=PCG(42, 54), out_f64=True, precision="f64")
    rgb64, hit64, stats64 = sc.render(p64, want_hit=True)
    assert stats64["precision_used"] == _abi.RT_PRECISION_F64
    assert np.array_equal(rgb64, rgb) and np.array_equal(hit64, hit) and stats64["rays_shadow"] == stats["rays_shadow"]
    # fp32 arithmetic: same image up to edge pixels
    p32 = make_params(size[0], size[1], cam, algo, s, aa_pcg=PCG(42, 54), precision="f32")
    rgb32, hit32, _ = sc.render(p32, want_hit=True)
    assert (hit32 != g[f"hit_s{s}"]).mean() < 2e-3
    assert_colors_close(rgb32, g[f"{algo}_s{s}_rgb"], rel=1e-4, frac_ok=0.995)


@pytest.mark.parametrize("tag", ["persp", "ortho"])
def test_scene2_deterministic_vs_reference(tag):
    fs, cam_p, cam_o = scene2_flat()
    cam = cam_p if tag == "persp" else cam_o
    g = golden("scene2.npz")
    sc = DeviceScene(fs)
    for algo in ("onoff", "flat", "pointlight"):
        p = make_params(96, 64, cam, algo, 0, background=(0.02, 0.03, 0.04), out_f64=True)
        rgb, hit, stats = sc.render(p, want_hit=True)
        assert np.array_equal(hit, g[f"{tag}_hit"]), algo
        assert np.allclose(rgb, g[f"{tag}_{algo}_rgb"], rtol=1e-11, atol=1e-14), algo
        assert stats["rays_shadow"] == int(g[f"{tag}_{algo}_rays_shadow"])


def test_config2_1080p_bit_exact_hit_index_and_colours():
    """BASELINE config 2: demo.txt, onoff + flat at 1920x1080, centre rays."""
    fs, cam = demo_flat()
    g = golden("demo_1080p.npz")
    sc = DeviceScene(fs)
    for algo in ("onoff", "flat", "pointlight"):
        rgb, hit, stats = sc.render(make_params(1920, 1080, cam, algo, 0), want_hit=True)
        assert np.array_equal(hit, g["hit"].astype(np.int32)), algo
        counts = np.bincount(hit.ravel() + 1, minlength=4)
        assert counts.tolist() == [484487, 518387, 1002874, 67852]
        assert np.allclose(rgb.astype(np.float64).reshape(-1, 3).mean(0), g[f"{algo}_mean"], rtol=1e-6)
        if algo == "flat":
            assert_colors_close(rgb, g["flat_rgb_f32"], rel=REL)
        elif algo == "pointlight":  # the reference's image is stored as a digest; the oracle renders it bit for bit
            want = oracle.render(fs, make_params(1920, 1080, cam, algo, 0), want_hit=False)["rgb"].astype(np.float32)
            assert sha256_of(want) == str(g["pointlight_rgb_f32_sha256"])
            assert_colors_close(rgb, want, rel=REL)
        assert [stats["rays_closest"], stats["rays_shadow"]] == g[f"{algo}_rays"].tolist()


# ------------------------------------------------------------------ hybrid precision (what AUTO resolves to)
def _assert_hybrid_is_fp64(sc, cam, w, h, algo, S, **kw):
    a, ha, sa = sc.render(make_params(w, h, cam, algo, S, aa_pcg=PCG(42, 54), out_f64=True, precision="f64", **kw), want_hit=True)
    b, hb, sb = sc.render(make_params(w, h, cam, algo, S, aa_pcg=PCG(42, 54), out_f64=True, precision="hybrid", **kw), want_hit=True)
    assert sb["precision_used"] == _abi.RT_PRECISION_HYBRID and sa["precision_used"] == _abi.RT_PRECISION_F64
    assert np.array_equal(ha, hb), (algo, S, int((ha != hb).sum()))
    assert np.array_equal(a, b), (algo, S, int((a != b).any(axis=-1).sum()))
    assert (sa["rays_closest"], sa["rays_shadow"], sa["samples"]) == (sb["rays_closest"], sb["rays_shadow"], sb["samples"])
    return sa, sb


@pytest.mark.parametrize("n_spheres", [0, 1, 3, 37, 1100])
def test_hybrid_gate_never_changes_the_fp64_image(n_spheres):
    """RT_PRECISION_HYBRID (rt_resolve_hybrid.cuh): the fp32 gate only decides which spheres the fp64 code
    looks at, and it is conservative — so hit index, colours (fp64 output) and shadow-ray counts must equal the
    plain fp64 kernel's BIT FOR BIT: every renderer, 1 / 4 / 9 samples per pixel (one ray per sweep, four
    per sweep, four with a remainder), odd image sizes, resident tables (<= 96 KB) and streamed ones
    (1 100 spheres x 2 origins: two chunks per sweep), row and strata partitions."""
    rs = scenes.random_spheres_scene(n_spheres, 2024, 4, 20.0, with_light=True)
    sc = DeviceScene(flatten_world(rs.world))
    w, h = (97, 61) if n_spheres > 100 else (67, 41)
    for algo in ("onoff", "flat", "pointlight"):
        for S in (0, 2, 3):
            _assert_hybrid_is_fp64(sc, rs.camera, w, h, algo, S)
    _assert_hybrid_is_fp64(sc, rs.camera, w, h, "pointlight", 2, part_mode=_abi.RT_PART_ROWS, part_rank=1, part_count=3)
    _assert_hybrid_is_fp64(sc, rs.camera, w, h, "pointlight", 2, part_mode=_abi.RT_PART_SPP, part_rank=1, part_count=2)


def test_hybrid_on_the_reference_scenes_and_awkward_geometry():
    """demo.txt and the second golden scene (ellipsoids, image pigment, two lights) through the hybrid path
    against the plain fp64 kernel; then geometry that stresses the gate's error bound: a camera inside a
    sphere, a light inside a sphere, needle- and pancake-shaped ellipsoids (condition number 1e3), a scene
    sitting 1e4 units from the world's origin (where the fp32 form M o + t has lost four digits), and spheres
    seen from 1e5 radii away.  An orthogonal camera has no common ray origin: AUTO stays on the fp64 kernel."""
    from pytracer_b200 import (Color, DiffuseBRDF, Material, PerspectiveCamera, Plane, Point, PointLight, Sphere,
                               UniformPigment, Vec, World, rotation_x, rotation_z, scaling, translation)

    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    for algo in ("onoff", "flat", "pointlight"):
        _assert_hybrid_is_fp64(sc, cam, 160, 120, algo, 2)
    fs2, cam_p, cam_o = scene2_flat()
    sc2 = DeviceScene(fs2)
    for algo in ("onoff", "flat", "pointlight"):
        _assert_hybrid_is_fp64(sc2, cam_p, 96, 64, algo, 2, background=(0.02, 0.03, 0.04))
    _, _, st = sc2.render(make_params(32, 24, cam_o, "flat", 0))
    assert st["precision_used"] == _abi.RT_PRECISION_F64
    with pytest.raises(Exception):
        sc2.render(make_params(32, 24, cam_o, "flat", 0, precision="hybrid"))

    mat = Material(DiffuseBRDF(UniformPigment(Color(0.5, 0.6, 0.7))), UniformPigment(Color(0.1, 0.0, 0.0)))
    for offset in (0.0, 1.0e4):
        base = translation(Vec(offset, -offset, 0.0))
        world = World()
        world.add_shape(Sphere(base * scaling(Vec(30.0, 30.0, 30.0)), mat))                       # the camera is inside
        world.add_shape(Sphere(base * translation(Vec(3.0, 0.0, 0.0)) * scaling(Vec(1e-3, 1.0, 1.0)), mat))  # pancake
        world.add_shape(Sphere(base * translation(Vec(4.0, 1.0, 0.5)) * rotation_z(33.0) * rotation_x(71.0) * scaling(Vec(2.0, 2e-3, 2e-3)), mat))  # needle
        world.add_shape(Sphere(base * translation(Vec(5.0, -1.0, 0.0)) * scaling(Vec(5e-5, 5e-5, 5e-5)), mat))  # 1e5 radii away
        world.add_shape(Sphere(base * translation(Vec(2.0, 2.0, 2.0)) * scaling(Vec(0.5, 0.5, 0.5)), mat))   # the light is inside
        for k in range(24):
            world.add_shape(Sphere(base * translation(Vec(3.0 + 0.3 * k, 0.1 * k - 1.0, 0.2 * (k % 5) - 0.4)) * rotation_z(10.0 * k)
                                   * scaling(Vec(0.05 + 0.01 * k, 0.3, 0.02 + 0.02 * (k % 7))), mat))
        world.add_shape(Plane(base * translation(Vec(0.0, 0.0, -1.0)), mat))
        world.add_light(PointLight(Point(offset + 2.0, -offset + 2.0, 2.0), Color(1.0, 1.0, 1.0)))
        world.add_light(PointLight(Point(offset + 0.0, -offset - 3.0, 4.0), Color(0.5, 0.5, 0.5), 1.0))
        cam = PerspectiveCamera(screen_distance=1.0, aspect_ratio=1.5, transformation=base * translation(Vec(-1.0, 0.0, 0.0)))
        sc3 = DeviceScene(world)
        for algo in ("onoff", "pointlight"):
            sa, _ = _assert_hybrid_is_fp64(sc3, cam, 150, 100, algo, 2)
        assert sa["rays_shadow"] > 0


def test_config5_full_size_hybrid_equals_fp64():
    """BASELINE config 5 at full size (4096 ellipsoids, pointlight, 3840x2160, 4 spp; 33.2 M samples):
    the default precision (AUTO -> hybrid) gives the fp64 kernel's frame bit for bit — all 8.3 M hit indices
    and 24.9 M colour values — several times faster, and a window of it equals the oracle."""
    rs = scenes.random_spheres_scene(4096, 2025, 5, 40.0, with_light=True)
    fs = flatten_world(rs.world)
    sc = DeviceScene(fs)
    a, ha, sa = sc.render(make_params(3840, 2160, rs.camera, "pointlight", 2, aa_pcg=PCG(42, 54), precision="f64"), want_hit=True)
    b, hb, sb = sc.render(make_params(3840, 2160, rs.camera, "pointlight", 2, aa_pcg=PCG(42, 54)), want_hit=True)
    assert sb["precision_used"] == _abi.RT_PRECISION_HYBRID
    assert np.array_equal(ha, hb) and np.array_equal(a, b)
    assert (sa["rays_closest"], sa["rays_shadow"]) == (sb["rays_closest"], sb["rays_shadow"])
    print(f"config 5: fp64 {sa['kernel_ms']:.1f} ms, hybrid {sb['kernel_ms']:.1f} ms ({sa['kernel_ms'] / sb['kernel_ms']:.2f}x)")
    assert sb["kernel_ms"] < 0.5 * sa["kernel_ms"]
    # fp32 against the same frame: the measured hit-index mismatch rate of the pure-fp32 kernels
    c, hc, _ = sc.render(make_params(3840, 2160, rs.camera, "pointlight", 2, aa_pcg=PCG(42, 54), precision="f32"), want_hit=True)
    d, hd, _ = sc.render(make_params(3840, 2160, rs.camera, "pointlight", 2, aa_pcg=PCG(42, 54), precision="f32", accel="bvh"), want_hit=True)
    print(f"config 5 fp32 hit-index mismatch vs fp64: linear {(hc != ha).mean():.2e}, bvh {(hd != ha).mean():.2e}, linear vs bvh {(hc != hd).mean():.2e}")
    assert (hc != ha).mean() < 5e-4 and (hd != ha).mean() < 5e-4


# ------------------------------------------------------------------ path tracing
def test_config1_replay_reproduces_the_reference_image():
    """BASELINE config 1 (demo.txt 160x120, 1 spp, N=10, depth 3, seeds 42/45): feeding the device
    the state the reference's single PCG stream has at the start of every sample reproduces the
    reference IMAGE (not just its distribution): fp64 to rounding, fp32 within 1e-4 for all but a
    handful of pixels where a discrete decision flips."""
    fs, cam = demo_flat()
    g = golden("demo_c1_pathtracing_160x120.npz")
    states = oracle.render(fs, c1_params(cam), want_states=True)["sample_states"]
    sc = DeviceScene(fs)
    p = c1_params(cam, rng_mode=_abi.RT_RNG_REPLAY, variant="mega", precision="f64", out_f64=True)
    rgb, _, stats = sc.render(p, replay_states=states)
    assert stats["rays_closest"] == int(g["rays_closest"]) == 393440
    assert np.allclose(rgb, g["rgb"], rtol=1e-9, atol=1e-12)
    p = c1_params(cam, rng_mode=_abi.RT_RNG_REPLAY, variant="mega", precision="f32")
    rgb32, _, stats32 = sc.render(p, replay_states=states)
    # fp32 walks the same tree as the fp64 reference: a ray that starts on a sphere uses the exact
    # second root for that sphere (rt_device.cuh: sphere_t_at), so the phantom re-hits fp32 would
    # otherwise see at t ~ 1e-4 on grazing mirror reflections (tmin = 1e-5 is tuned for fp64) are gone.
    assert abs(stats32["rays_closest"] - 393440) <= 40
    assert_colors_close(rgb32, g["rgb"], rel=1e-3, frac_ok=0.9995)
    assert np.allclose(rgb32.reshape(-1, 3).mean(0), g["rgb"].reshape(-1, 3).mean(0), rtol=2e-3)


def test_replay_with_roulette_inside_the_tree():
    fs, cam = demo_flat()
    g = golden("demo_pt_small.npz")
    args = dict(algorithm="pathtracing", samples_per_side=2, num_of_rays=3, max_depth=5, rr_limit=2,
                aa_pcg=PCG(7, 11), pt_pcg=PCG(99, 3), background=(0.05, 0.02, 0.01))
    states = oracle.render(fs, make_params(40, 30, cam, **args), want_states=True)["sample_states"]
    sc = DeviceScene(fs)
    p = make_params(40, 30, cam, rng_mode=_abi.RT_RNG_REPLAY, variant="mega", precision="f64", out_f64=True, **args)
    rgb, _, stats = sc.render(p, replay_states=states)
    assert stats["rays_closest"] == int(g["rays_closest"])
    assert np.allclose(rgb, g["rgb"], rtol=1e-9, atol=1e-12)


def _oracle_runs(fs, params_fn, runs):
    """K independent oracle renders (own jitter and scatter streams each; rows spread over the host's threads).
    Returns (images, rays per sample)."""
    import os

    threads = max(1, min(32, os.cpu_count() or 1))
    imgs, rays, samples = [], 0, 0
    for k in range(runs):
        r = oracle.render_threaded(fs, params_fn(PCG(1000 + k, 7), PCG(2000 + k, 9)), threads)
        imgs.append(r["rgb"].copy())
        rays += r["rays_closest"]
        samples += r["samples"]
    return np.stack(imgs), rays / samples


@pytest.mark.parametrize("variant", ["warp", "mega"])
def test_streams_agree_statistically_with_the_reference_estimator(variant):
    """demo.txt 160x120, N=10, depth 3: the GPU at 1024 spp against 24 independent 16-spp oracle renders.
    Bars (north star): every per-pixel mean within 3 sigma of the Monte Carlo error — evaluated against
    Student's t because sigma is estimated from the 24 runs (util.mc_agreement) — and image-mean luminance
    within 0.5 %."""
    fs, cam = demo_flat()
    args = dict(algorithm="pathtracing", num_of_rays=10, max_depth=3, rr_limit=3)
    ref, ref_rays = _oracle_runs(fs, lambda aa, pt: make_params(160, 120, cam, samples_per_side=4, aa_pcg=aa, pt_pcg=pt, **args), runs=24)
    ref_mean = ref.mean(0)
    sc = DeviceScene(fs)
    p = make_params(160, 120, cam, samples_per_side=32, aa_pcg=PCG(11, 3), pt_pcg=PCG(77, 5), variant=variant, **args)
    rgb, _, stats = sc.render(p)
    assert stats["variant_used"] == _abi.VARIANTS[variant] and stats["overflow"] == 0
    gpu = rgb.astype(np.float64)
    assert_luminance_agreement(gpu, ref, what=f"demo.txt 160x120 {variant}")
    assert abs(luminosity(ref_mean).mean() - 0.29537) < 0.005 * 0.29537  # BASELINE.md anchor
    assert_mc_agreement(gpu, ref, samples_ratio=(24 * 16) / 1024.0, n_ref=24 * 16, what=f"demo.txt 160x120 {variant}")
    # rays per sample as the reference counts them (BASELINE.md: 20.49 per sample)
    assert abs(stats["rays_closest"] / stats["samples"] - ref_rays) < 0.005 * ref_rays and abs(ref_rays - 20.49) < 0.1


def test_warp_and_mega_agree_on_scene2_with_deep_roulette():
    fs, cam_p, _ = scene2_flat()
    sc = DeviceScene(fs)
    args = dict(algorithm="pathtracing", samples_per_side=6, num_of_rays=3, max_depth=5, rr_limit=2,
                background=(0.02, 0.03, 0.04))
    imgs = {}
    for variant in ("warp", "mega"):
        rgb, _, stats = sc.render(make_params(48, 32, cam_p, aa_pcg=PCG(3, 1), pt_pcg=PCG(4, 1), variant=variant, **args))
        assert stats["overflow"] == 0
        imgs[variant] = rgb.astype(np.float64)
    ref = np.stack([oracle.render(fs, make_params(48, 32, cam_p, aa_pcg=PCG(50 + k, 1), pt_pcg=PCG(60 + k, 1), **args),
                                  want_hit=False)["rgb"] for k in range(6)])
    ref_mean = ref.mean(0)
    for variant, img in imgs.items():
        assert abs(luminosity(img).mean() - luminosity(ref_mean).mean()) < 0.01 * luminosity(ref_mean).mean(), variant
        assert np.allclose(img.reshape(-1, 3).mean(0), ref_mean.reshape(-1, 3).mean(0), rtol=2e-2), variant


def test_furnace():
    """tests/test_all.py:1014-1051: inside an emissive diffuse sphere L = Le / (1 - rho)."""
    from pytracer_b200 import Color, DiffuseBRDF, Material, Point, Ray, Sphere, UniformPigment, Vec, World
    from pytracer_b200.render import PathTracer

    a = golden("analytic.npz")
    pcg = PCG()
    for i in range(5):
        emitted, refl = pcg.random_float(), pcg.random_float() * 0.9
        assert (emitted, refl) == tuple(a["furnace"][i][:2])
        world = World()
        world.add_shape(Sphere(material=Material(DiffuseBRDF(UniformPigment(Color(refl, refl, refl))),
                                                 UniformPigment(Color(emitted, emitted, emitted)))))
        tracer = PathTracer(pcg=pcg, num_of_rays=1, world=world, max_depth=100, russian_roulette_limit=101)
        color = tracer(Ray(origin=Point(0, 0, 0), dir=Vec(1, 0, 0)))
        expected = emitted / (1.0 - refl)
        assert abs(color.r - expected) < 1e-3 and abs(color.g - expected) < 1e-3 and abs(color.b - expected) < 1e-3
        assert np.allclose(color.rgb(), a["furnace"][i][2:5], rtol=1e-9)  # the reference's own run
        assert pcg.state == int(a[f"furnace_state1_{i}"])              # generator left where the reference leaves it
        # warp variant: one pixel, 64 spp, same analytic answer
        from pytracer_b200 import HdrImage, OrthogonalCamera
        from pytracer_b200.imagetracer import CudaImageTracer
        tracer_w = PathTracer(pcg=PCG(5, i), num_of_rays=1, world=world, max_depth=100, russian_roulette_limit=101, variant="warp")
        img = HdrImage(2, 2)
        cam = OrthogonalCamera(transformation=__import__("pytracer_b200").scaling(Vec(0.1, 0.1, 0.1)))
        CudaImageTracer(img, cam, samples_per_side=3).fire_all_rays(tracer_w)
        assert np.allclose(img.rgb_array(), expected, rtol=1e-3)


def test_point_light_renderer_analytic():
    """tests/test_all.py:1054-1116 restated: ambient + emitted + rho cos(45 deg) / pi."""
    import math
    from pytracer_b200 import (Color, DiffuseBRDF, Material, Plane, Point, PointLight, Ray, UniformPigment,
                               Vec, World)
    from pytracer_b200.render import PointLightRenderer

    world = World()
    world.add_shape(Plane(material=Material(DiffuseBRDF(UniformPigment(Color(0.2, 0.4, 0.6))), UniformPigment(Color(0.01, 0.02, 0.03)))))
    world.add_light(PointLight(Point(-1.0, 0.0, 1.0), Color(1.0, 1.0, 1.0)))
    renderer = PointLightRenderer(world=world, ambient_color=Color(0.1, 0.1, 0.1))
    color = renderer(Ray(origin=Point(0.0, 0.0, 1.0), dir=Vec(0.0, 0.0, -1.0)))
    cos45 = math.cos(math.pi / 4)
    for got, rho, em in zip(color.rgb(), (0.2, 0.4, 0.6), (0.01, 0.02, 0.03)):
        assert abs(got - (0.1 + em + rho / math.pi * cos45)) < 1e-5 * got


def test_partitions_sum_to_the_unpartitioned_image():
    """The multi-GPU contract: every rank's share summed over ranks is the 1-GPU image."""
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    base = dict(algorithm="pathtracing", samples_per_side=4, num_of_rays=10, max_depth=3, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54))
    for variant in ("warp", "mega"):
        full, _, st_full = sc.render(make_params(96, 72, cam, variant=variant, **base))
        for count in (2, 8):
            acc = np.zeros_like(full, dtype=np.float64)
            rays = 0
            for rank in range(count):
                part, _, st = sc.render(make_params(96, 72, cam, variant=variant, part_mode=_abi.RT_PART_SPP,
                                                    part_rank=rank, part_count=count, **base))
                acc += part
                rays += st["rays_closest"]
            assert rays == st_full["rays_closest"]
            # different kernel instantiations round differently in the last bit; a ray grazing a
            # silhouette may then fall on the other side, so a handful of pixels are allowed to differ
            close = np.isclose(acc, full, rtol=2e-5, atol=1e-6)
            assert close.mean() > 0.9995, (variant, count, int((~close).sum()))
    p_full = make_params(97, 61, cam, "pointlight", 2, aa_pcg=PCG(42, 54))
    full, hit_full, _ = sc.render(p_full, want_hit=True)
    acc = np.zeros_like(full)
    for rank in range(3):
        part, hit, _ = sc.render(make_params(97, 61, cam, "pointlight", 2, aa_pcg=PCG(42, 54), part_mode=_abi.RT_PART_ROWS,
                                             part_rank=rank, part_count=3), want_hit=True)
        acc += part
        assert np.array_equal(hit[rank::3], hit_full[rank::3])
    assert np.array_equal(acc, full)  # disjoint rows: x + 0 is exact


def test_many_shapes_chunked_scan_and_textures():
    """More shapes than one shared-memory chunk holds (fp64: 96 KB / 96 B = 1024): the chunked
    block-synchronous sweep must pick the same winners as the oracle's plain loop."""
    rs = scenes.random_spheres_scene(1100, 2024, 4, 20.0, with_light=True)
    fs = flatten_world(rs.world)
    sc = DeviceScene(fs)
    for algo in ("flat", "pointlight"):
        p = make_params(64, 36, rs.camera, algo, 0, out_f64=True)
        ref = oracle.render(fs, p)
        rgb, hit, stats = sc.render(p, want_hit=True)
        assert np.array_equal(hit, ref["hit_index"]), algo
        assert np.allclose(rgb, ref["rgb"], rtol=1e-9, atol=1e-12), algo
        assert stats["rays_shadow"] == ref["rays_shadow"]
        rgb32, hit32, _ = sc.render(make_params(64, 36, rs.camera, algo, 0, precision="f32"), want_hit=True)
        assert (hit32 != ref["hit_index"]).mean() < 5e-3
    # path tracing on the same scene, statistical (north-star bars; the full-size frame is config 4's test)
    args = dict(algorithm="pathtracing", num_of_rays=4, max_depth=2)
    ref, ref_rays = _oracle_runs(fs, lambda aa, pt: make_params(32, 18, rs.camera, samples_per_side=4, aa_pcg=aa, pt_pcg=pt, **args), runs=16)
    for variant in ("warp", "mega"):
        rgb, _, stats = sc.render(make_params(32, 18, rs.camera, samples_per_side=32, variant=variant, **args))
        assert stats["overflow"] == 0
        assert_luminance_agreement(rgb, ref, what=f"1100 spheres 32x18 {variant}")
        assert_mc_agreement(rgb, ref, samples_ratio=256.0 / 1024.0, n_ref=256, what=f"1100 spheres 32x18 {variant}")
        assert abs(stats["rays_closest"] / stats["samples"] - ref_rays) < 0.01 * ref_rays


def test_empty_world_and_edge_sizes():
    from pytracer_b200 import World
    from pytracer_b200.scene import PerspectiveCamera

    sc = DeviceScene(World())
    for algo in ("onoff", "flat", "pointlight", "pathtracing"):
        rgb, hit, stats = sc.render(make_params(5, 3, PerspectiveCamera(), algo, 1, background=(0.25, 0.5, 0.75), num_of_rays=2, max_depth=2), want_hit=True)
        assert np.allclose(rgb, [0.25, 0.5, 0.75]) and (hit == -1).all()
        assert stats["rays_closest"] == 15
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    rgb, hit, _ = sc.render(make_params(1, 1, cam, "flat", 0), want_hit=True)
    assert rgb.shape == (1, 1, 3)
    with pytest.raises(Exception):
        sc.render(make_params(0, 4, cam, "flat", 0))


DEMO_TEXT = '''
float clock(150)
material sky_material(diffuse(uniform(<0, 0, 0>)), uniform(<0.7, 0.5, 1>))
material ground_material(diffuse(checkered(<0.3, 0.5, 0.1>, <0.1, 0.2, 0.5>, 4)), uniform(<0, 0, 0>))
material sphere_material(specular(uniform(<0.5, 0.5, 0.5>)), uniform(<0, 0, 0>))
point_light([10, 10, 10], <1, 1, 1>, 1)
plane (sky_material, translation([0, 0, 100]) * rotation_y(clock))
plane (ground_material, identity)
sphere(sphere_material, translation([0, 0, 1]))
camera(perspective, rotation_z(30) * translation([-4, 0, 1]), 1.0, 1.0)
'''


def test_render_command_writes_the_reference_image(tmp_path):
    """`render --algorithm flat` (the reference's CLI options, main.py:76-129) -> PFM == golden."""
    from click.testing import CliRunner

    from pytracer_b200.hdrimage import read_pfm_image
    from pytracer_b200.main import cli

    scene_file = tmp_path / "demo.txt"
    scene_file.write_text(DEMO_TEXT)
    pfm, png = tmp_path / "out.pfm", tmp_path / "out.png"
    res = CliRunner().invoke(cli, ["render", "--width", "160", "--height", "120", "--algorithm", "flat",
                                   "--samples-per-pixel", "0", "--pfm-output", str(pfm), "--png-output", str(png),
                                   "--parser", "builtin", str(scene_file)])
    assert res.exit_code == 0, res.output
    assert "Using flat renderer" in res.output
    with open(pfm, "rb") as f:
        img = read_pfm_image(f)
    g = golden("demo_deterministic.npz")
    assert np.array_equal(img.rgb_array(), g["flat_s0_rgb"].astype(np.float32))
    assert png.exists() and png.stat().st_size > 100
    res = CliRunner().invoke(cli, ["render", "--samples-per-pixel", "3", str(scene_file)])
    assert "must be a perfect square" in res.output
    res = CliRunner().invoke(cli, ["render", "--width", "64", "--height", "48", "--samples-per-pixel", "4",
                                   "--pfm-output", str(pfm), "--png-output", str(png), str(scene_file)])
    assert res.exit_code == 0 and "Using a path tracer" in res.output


# ------------------------------------------------------------------ BASELINE sizes, size-independent properties
def test_config3_full_size_properties():
    """BASELINE config 3 (demo.txt 1920x1080, 64 spp, N=10, depth 3) at full size.  The reference needs
    ~40 core-hours for this frame, so the check goes through properties the domain offers:
      * the expectation does not depend on resolution: image-mean RGB / luminance equal the converged
        reference anchors of BASELINE.md (0.5 % bar of the north star);
      * the camera's aspect ratio comes from the scene, so a 12x9 box-downsample of the 1080p frame has
        exactly the pixel footprints of a 160x120 render: compare it per pixel with oracle statistics;
      * rays per sample as the reference counts them (20.5, SURVEY §8a);
      * the image does not depend on how samples are spread over GPUs (strata of 8 ranks summed)."""
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    args = dict(algorithm="pathtracing", samples_per_side=8, num_of_rays=10, max_depth=3, rr_limit=3,
                aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54))
    rgb, _, stats = sc.render(make_params(1920, 1080, cam, **args))
    assert stats["samples"] == 1920 * 1080 * 64 and stats["overflow"] == 0
    assert abs(stats["rays_closest"] / stats["samples"] - 20.5) < 0.1
    img = rgb.astype(np.float64)
    mean_rgb = img.reshape(-1, 3).mean(0)
    assert np.allclose(mean_rgb, [0.243146, 0.207565, 0.393151], rtol=5e-3)   # BASELINE.md §2 anchors
    assert abs(luminosity(img).mean() - 0.29537) < 0.005 * 0.29537
    small = img.reshape(120, 9, 160, 12, 3).mean(axis=(1, 3))                   # 12x9 box filter -> 160x120
    ref, _ = _oracle_runs(fs, lambda aa, pt: make_params(160, 120, cam, algorithm="pathtracing", samples_per_side=4, num_of_rays=10,
                                                         max_depth=3, aa_pcg=aa, pt_pcg=pt), runs=24)
    # the downsampled frame carries 6912 samples per footprint against the oracle's 384
    assert_mc_agreement(small, ref, samples_ratio=384.0 / 6912.0, n_ref=384, what="config 3, 12x9 footprints")
    assert_luminance_agreement(small, ref, what="config 3, 12x9 footprints")
    acc = np.zeros_like(img)
    for rank in range(8):
        part, _, st = sc.render(make_params(1920, 1080, cam, part_mode=_abi.RT_PART_SPP, part_rank=rank, part_count=8, **args))
        acc += part
    close = np.isclose(acc, img, rtol=5e-5, atol=2e-6)
    assert close.mean() > 0.9999


def test_config4_full_size_properties():
    """BASELINE config 4 at its stated size: 1 024 randomly transformed ellipsoids + 2 planes, checkered and
    image pigments, diffuse and mirror surfaces, path tracing 3840x2160 at 16 spp (132.7 M samples, ~127 rays
    per sample) — the frame where the chunked pair sweep, the candidate lists, the half-warp split and the
    texture unit all run together.  The reference needs ~10^4 core-hours for it, so, like config 3:
      * the camera's aspect ratio comes from the scene, so a 120x120 box-downsample of the 4K frame has exactly
        the pixel footprints of a 32x18 render: per footprint, the mean must lie within 3 sigma of the
        Monte Carlo error of 16 independent 16-spp oracle renders (threaded over rows; ~19 M rays against
        1 026 shapes, about a minute of host time), and the image-mean luminance within 0.5 %
        (north-star bars; render.py:99-139, materials.py:62-100);
      * rays per sample equal the oracle's count;
      * the strata shares of 8 ranks sum to the single-GPU frame;
      * the sphere hierarchy (accel="bvh") traces the same tree: ray counts and footprints agree."""
    rs = scenes.random_spheres_scene(1024, 2024, 4, 20.0)
    fs = flatten_world(rs.world)
    sc = DeviceScene(fs)
    args = dict(algorithm="pathtracing", samples_per_side=4, num_of_rays=10, max_depth=3, rr_limit=3,
                aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54))
    rgb, _, stats = sc.render(make_params(3840, 2160, rs.camera, **args))
    assert stats["samples"] == 3840 * 2160 * 16 and stats["overflow"] == 0 and stats["variant_used"] == _abi.RT_VARIANT_WARP
    img = rgb.astype(np.float64)
    small = img.reshape(18, 120, 32, 120, 3).mean(axis=(1, 3))
    ref, ref_rays = _oracle_runs(fs, lambda aa, pt: make_params(32, 18, rs.camera, algorithm="pathtracing", samples_per_side=4,
                                                                num_of_rays=10, max_depth=3, rr_limit=3, aa_pcg=aa, pt_pcg=pt), runs=16)
    ratio = 256.0 / (120 * 120 * 16)
    assert_luminance_agreement(small, ref, what="config 4, 120x120 footprints")
    assert_mc_agreement(small, ref, samples_ratio=ratio, n_ref=256, what="config 4, 120x120 footprints")
    rays_gpu = stats["rays_closest"] / stats["samples"]
    print(f"config 4: rays per sample GPU {rays_gpu:.2f}, oracle {ref_rays:.2f}; kernel {stats['kernel_ms']:.0f} ms")
    assert abs(rays_gpu - ref_rays) < 0.01 * ref_rays
    # the same bars on a four times finer grid, 64x36 footprints of 60x60 pixels (6 912 values), against the
    # committed oracle statistics (tests/golden/make_golden_c4.py: 16 runs x 16 spp, 75 M oracle rays)
    fix = golden("c4_oracle_64x36.npz")
    fine = img.reshape(36, 60, 64, 60, 3).mean(axis=(1, 3))
    fine_ratio = 256.0 / (60 * 60 * 16)
    assert_luminance_agreement(fine, fix["runs"], what="config 4, 60x60 footprints")
    assert_mc_agreement(fine, fix["runs"], samples_ratio=fine_ratio, n_ref=256, what="config 4, 60x60 footprints")
    assert abs(rays_gpu - float(fix["rays_per_sample"])) < 0.01 * float(fix["rays_per_sample"])
    # strata split over 8 ranks (2 strata each) sums to the frame
    acc = np.zeros_like(img)
    rays = 0
    for rank in range(8):
        part, _, st = sc.render(make_params(3840, 2160, rs.camera, part_mode=_abi.RT_PART_SPP, part_rank=rank, part_count=8, **args))
        acc += part
        rays += st["rays_closest"]
    assert abs(rays - stats["rays_closest"]) <= 1e-5 * rays
    close = np.isclose(acc, img, rtol=5e-5, atol=2e-6)
    assert close.mean() > 0.999, close.mean()
    # the hierarchy walks the same ray tree
    rgb_b, _, st_b = sc.render(make_params(3840, 2160, rs.camera, accel="bvh", **args))
    assert st_b["overflow"] == 0
    assert abs(st_b["rays_closest"] - stats["rays_closest"]) <= 1e-4 * stats["rays_closest"]
    small_b = rgb_b.astype(np.float64).reshape(18, 120, 32, 120, 3).mean(axis=(1, 3))
    assert np.allclose(small_b, small, rtol=2e-3, atol=1e-4)
    assert_luminance_agreement(small_b, ref, what="config 4 bvh, 120x120 footprints")
    assert_mc_agreement(small_b, ref, samples_ratio=ratio, n_ref=256, what="config 4 bvh, 120x120 footprints")
    fine_b = rgb_b.astype(np.float64).reshape(36, 60, 64, 60, 3).mean(axis=(1, 3))
    assert_mc_agreement(fine_b, fix["runs"], samples_ratio=fine_ratio, n_ref=256, what="config 4 bvh, 60x60 footprints")


def test_config5_full_size_properties():
    """BASELINE config 5 (4096 ellipsoids, pointlight, 3840x2160, 4 spp) at full size in fp32, checked
    through properties: interleaved-row shares of 8 ranks sum bit-exactly to the single-GPU frame
    (x + 0 is exact), every sample traces one primary ray and at most one shadow ray, and a 96x54
    window re-rendered on its own in fp64 against the oracle agrees on the hit index bit for bit."""
    rs = scenes.random_spheres_scene(4096, 2025, 5, 40.0, with_light=True)
    fs = flatten_world(rs.world)
    sc = DeviceScene(fs)
    p = make_params(3840, 2160, rs.camera, "pointlight", 2, aa_pcg=PCG(42, 54), precision="f32")
    full, _, stats = sc.render(p)
    n = 3840 * 2160 * 4
    assert stats["samples"] == stats["rays_closest"] == n and 0 < stats["rays_shadow"] <= n
    acc = np.zeros_like(full)
    shadow = 0
    for rank in range(8):
        part, _, st = sc.render(make_params(3840, 2160, rs.camera, "pointlight", 2, aa_pcg=PCG(42, 54), precision="f32",
                                            part_mode=_abi.RT_PART_ROWS, part_rank=rank, part_count=8))
        acc += part
        shadow += st["rays_shadow"]
    assert np.array_equal(acc, full) and shadow == stats["rays_shadow"]
    small = make_params(96, 54, rs.camera, "pointlight", 0, out_f64=True)
    ref = oracle.render(fs, small)
    rgb64, hit64, st64 = sc.render(small, want_hit=True)
    assert np.array_equal(hit64, ref["hit_index"]) and st64["rays_shadow"] == ref["rays_shadow"]
    assert np.allclose(rgb64, ref["rgb"], rtol=1e-9, atol=1e-12)


# ------------------------------------------------------------------ tone mapping (SURVEY §8f-2)
def test_tone_mapping_matches_the_reference_bytes():
    """hdrimages.py:120-171 on the device: LDR bytes bit-exact against the reference's PNG, average
    luminosity and normalised values to fp64 / fp32 rounding."""
    from pytracer_b200 import tonemap
    from test_oracle_golden import tonemap_cases

    for i, img, factor, lum, gamma, g in tonemap_cases():
        avg = tonemap.average_luminosity(img)
        assert abs(avg - float(g[f"case{i}_avg"])) <= 1e-10 * avg  # order of the fp64 sum only
        hdr, ldr, st = tonemap.tone_map(img, factor, lum, gamma)
        assert np.array_equal(ldr, g[f"case{i}_ldr"]), f"case {i}: {(ldr != g[f'case{i}_ldr']).sum()} bytes differ"
        assert np.allclose(hdr, g[f"case{i}_hdr"], rtol=2e-7, atol=1e-45)  # stored as fp32
        assert abs(st["luminosity"] - (lum if lum else float(g[f"case{i}_avg"]))) <= 1e-10 * st["luminosity"]
        assert st["n_launches"] == (1 if lum else 2)


def test_tone_mapping_without_clamp_saturates_like_the_reference():
    """HdrImage.write_ldr_image alone (flags = 0) and normalize_image + write_ldr_image (no clamp_image) on
    channels above 1: int(255 c) exceeds 255 and PIL's putpixel clips it (hdrimages.py:160-165), so the byte
    is 255 — in the fp32 fast path (gamma 1, LDR only) as in the exact one (gamma != 1, HDR requested)."""
    from pytracer_b200 import tonemap

    rng = np.random.default_rng(3)
    img = (10.0 ** rng.uniform(-3.0, 1.5, size=(64, 96, 3))).astype(np.float32)
    img[0, 0] = (1.004, 1.5, 300.0)
    img[0, 1] = (255.5 / 255.0, 256.0 / 255.0, 1.0)
    for flags, factor, lum in ((0, 1.0, 1.0), (tonemap.NORMALIZE, 0.8, 0.5)):
        x = img.astype(np.float64) * ((factor / lum) if flags else 1.0)
        for gamma in (1.0, 2.2):
            want = np.clip((255.0 * (x if gamma == 1.0 else np.power(x, 1.0 / gamma))).astype(np.int64), 0, 255).astype(np.uint8)
            _, ldr, _ = tonemap.tone_map(img, factor, lum, gamma, want_hdr=False, flags=flags)
            assert np.array_equal(ldr, want), (flags, gamma, int((ldr != want).sum()))
            assert (want == 255).mean() > 0.2  # the case is exercised
        _, ldr2, _ = tonemap.tone_map(img, factor, lum, 1.0, want_hdr=True, flags=flags)  # exact kernel
        assert np.array_equal(ldr2, np.clip((255.0 * x).astype(np.int64), 0, 255).astype(np.uint8))


def test_renderer_reads_the_world_live():
    """The reference's renderers read World at every call (render.py:52-193), so editing a shape in place
    between two images must show: transformations are patched into the resident scene, anything else
    rebuilds it — never a stale image."""
    from pytracer_b200 import Color, HdrImage, Vec, translation
    from pytracer_b200.imagetracer import CudaImageTracer
    from pytracer_b200.render import FlatRenderer

    world, camera = scenes.demo_scene()
    renderer = FlatRenderer(world)

    def shoot(r):
        image = HdrImage(96, 72)
        CudaImageTracer(image, camera, samples_per_side=0).fire_all_rays(r)
        return image.rgb_array().copy()

    first = shoot(renderer)
    resident = renderer._scene
    assert np.array_equal(first, shoot(renderer)) and renderer._scene is resident      # unchanged: reused
    world.shapes[2].transformation = translation(Vec(0.0, 0.5, 1.2))                     # moved: patched in place
    moved = shoot(renderer)
    assert renderer._scene is resident and not np.array_equal(moved, first)
    assert np.array_equal(moved, shoot(FlatRenderer(world)))
    world.shapes[2].material.brdf.pigment.color = Color(0.9, 0.1, 0.1)                   # recoloured: rebuilt
    recoloured = shoot(renderer)
    assert renderer._scene is not resident and not np.array_equal(recoloured, moved)
    assert np.array_equal(recoloured, shoot(FlatRenderer(world)))


def test_hdrimage_tone_mapping_methods_mirror_the_reference():
    # tests/test_all.py:239-268 on the device-backed HdrImage
    from pytracer_b200.hdrimage import HdrImage
    from pytracer_b200.scene import Color

    def fresh():
        img = HdrImage(2, 1)
        img.set_pixel(0, 0, Color(0.5e1, 1.0e1, 1.5e1))
        img.set_pixel(1, 0, Color(0.5e3, 1.0e3, 1.5e3))
        return img

    assert abs(fresh().average_luminosity(delta=0.0) - 100.0) < 1e-9
    img = fresh()
    img.normalize_image(factor=1000.0, luminosity=100.0)
    assert img.get_pixel(0, 0).is_close(Color(0.5e2, 1.0e2, 1.5e2))
    assert img.get_pixel(1, 0).is_close(Color(0.5e4, 1.0e4, 1.5e4))
    img = fresh()
    img.clamp_image()
    for p in img.pixels:
        assert 0 <= p.r <= 1 and 0 <= p.g <= 1 and 0 <= p.b <= 1
    assert abs(img.get_pixel(0, 0).r - 5.0 / 6.0) < 1e-6


def test_tone_mapping_full_size_properties_on_device_buffers():
    """3840x2160 (BASELINE configs 4/5 frame size) on device buffers: the oracle on a window, and
    size-independent properties — scaling the image scales its average luminosity, a passed-in
    luminosity gives the same bytes as the computed one, the map is monotonic."""
    import torch

    from oracle import tonemap_oracle as tm
    from pytracer_b200 import tonemap

    h, w = 2160, 3840
    gen = torch.Generator(device="cuda").manual_seed(7)
    img = torch.exp(torch.randn((h, w, 3), device="cuda", generator=gen) * 2.0).contiguous()
    n = h * w
    ldr = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
    hdr = torch.empty_like(img)
    st = tonemap.tone_map_device(img.data_ptr(), n, 0.7, None, 1.0, hdr.data_ptr(), ldr.data_ptr())
    host = img.cpu().numpy()
    ref_lum = tm.average_luminosity(host)
    assert abs(st["luminosity"] - ref_lum) <= 1e-10 * ref_lum
    _, ref_hdr, ref_ldr = tm.tone_map(host[:64], 0.7, st["luminosity"], 1.0)
    assert np.array_equal(ldr[:64].cpu().numpy(), ref_ldr)
    assert np.allclose(hdr[:64].cpu().numpy(), ref_hdr, rtol=2e-7)
    # idempotence: passing the luminosity in skips the first kernel and gives the same bytes
    ldr2 = torch.empty_like(ldr)
    st2 = tonemap.tone_map_device(img.data_ptr(), n, 0.7, st["luminosity"], 1.0, 0, ldr2.data_ptr())
    assert st2["n_launches"] == 1 and torch.equal(ldr, ldr2)
    # homogeneity (delta = 1e-10 is negligible against exp(N(0, 2)) values)
    st4 = tonemap.tone_map_device((img * 4.0).contiguous().data_ptr(), n, 0.7, None, 1.0, 0, ldr2.data_ptr())
    assert abs(st4["luminosity"] / st["luminosity"] - 4.0) < 1e-6
    assert torch.equal(ldr, ldr2)  # same normalised image -> same bytes
    # monotonic: brighter input never gives a darker byte
    order = torch.argsort(img.reshape(-1)[: 1 << 20])
    b = ldr.reshape(-1)[: 1 << 20][order].to(torch.int16)
    assert int((b[1:] - b[:-1]).min()) >= 0
    # a misaligned view takes the scalar path and agrees
    flat = torch.empty(3 * n + 1, dtype=torch.float32, device="cuda")
    flat[1:] = img.reshape(-1)
    ldr3 = torch.empty(3 * n + 1, dtype=torch.uint8, device="cuda")
    tonemap.tone_map_device(flat.data_ptr() + 4, n, 0.7, st["luminosity"], 1.0, 0, ldr3.data_ptr() + 1)
    assert torch.equal(ldr3[1:], ldr.reshape(-1))


# ------------------------------------------------------------------ animation (SURVEY §8f-4)
def test_transform_updates_equal_a_rebuilt_scene():
    """rt_scene_update_transforms on a resident scene gives, bit for bit, the images of scenes built
    from scratch for the same frame (fp64 flat/pointlight + hit index, fp32 tables through the path
    tracer), on demo.txt's `clock` animation and on a many-sphere scene (packed pair table)."""
    from pytracer_b200.scene import Transformation, Vec, rotation_z, scaling, translation

    w0, cam = scenes.demo_scene(clock=150.0)
    resident = DeviceScene(w0)
    camera = flatten_camera(cam)
    for clock in (10.0, 275.0):
        w1, _ = scenes.demo_scene(clock=clock)
        w1.shapes[2].transformation = translation(Vec(0.3, -0.2, 1.0 + clock / 1000.0)) * scaling(Vec(1.0, 0.7, 1.2))
        fresh = DeviceScene(w1)
        resident.update_from_world(w1)
        for algo in ("flat", "pointlight"):
            p = make_params(96, 72, camera, algo, 2, aa_pcg=PCG(42, 54))
            a, ha, _ = resident.render(p, want_hit=True)
            b, hb, _ = fresh.render(p, want_hit=True)
            assert np.array_equal(a, b) and np.array_equal(ha, hb), (clock, algo)
        p = make_params(64, 48, camera, "pathtracing", 2, num_of_rays=3, max_depth=3, rr_limit=2, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54))
        assert np.array_equal(resident.render(p)[0], fresh.render(p)[0]), clock
        fresh.close()
    # partial update of a scene with an odd number of spheres and planes in between
    rs = scenes.random_spheres_scene(37, 7, 3, 10.0)
    resident = DeviceScene(rs.world)
    camera = flatten_camera(rs.camera)
    moved = rs.world.shapes[5:12]
    for k, shape in enumerate(moved):
        shape.transformation = translation(Vec(0.1 * k, -0.2, 0.05 * k)) * shape.transformation * rotation_z(10.0 * k)
    fresh = DeviceScene(rs.world)
    flat = flatten_world(rs.world)
    resident.update_transforms(5, flat.shape_m.reshape(-1, 12)[5:12], flat.shape_invm.reshape(-1, 12)[5:12])
    for algo, prec in (("flat", "f64"), ("flat", "f32"), ("pathtracing", "f32")):
        p = make_params(80, 45, camera, algo, 1, num_of_rays=2, max_depth=2, aa_pcg=PCG(1, 2), pt_pcg=PCG(3, 4), precision=prec)
        assert np.array_equal(resident.render(p)[0], fresh.render(p)[0]), (algo, prec)
    with pytest.raises(Exception):
        resident.update_transforms(len(rs.world.shapes) - 1, np.zeros((2, 12)), np.zeros((2, 12)))


def test_animate_command_patches_the_resident_scene(tmp_path):
    """`animate` over demo.txt's clock: every frame equals a standalone `render -d clock:VALUE` of the
    same frame, and frames after the first are patched in place rather than rebuilt."""
    from click.testing import CliRunner

    from pytracer_b200.hdrimage import read_pfm_image
    from pytracer_b200.main import cli

    scene_file = tmp_path / "demo.txt"
    scene_file.write_text(DEMO_TEXT)
    prefix = str(tmp_path / "f")
    common = ["--width", "96", "--height", "72", "--algorithm", "pointlight", "--samples-per-pixel", "4", "--parser", "builtin"]
    res = CliRunner().invoke(cli, ["animate", *common, "--frames", "3", "--start", "0", "--stop", "90", "--output-prefix", prefix,
                                   str(scene_file)])
    assert res.exit_code == 0, res.output
    assert "patched in place for 2 of them" in res.output
    for f, clock in enumerate((0.0, 30.0, 60.0)):
        pfm = tmp_path / f"single{f}.pfm"
        res = CliRunner().invoke(cli, ["render", *common, "-d", f"clock:{clock}", "--pfm-output", str(pfm),
                                       "--png-output", str(tmp_path / "single.png"), str(scene_file)])
        assert res.exit_code == 0, res.output
        with open(pfm, "rb") as a, open(f"{prefix}{f:03d}.pfm", "rb") as b:
            assert np.array_equal(read_pfm_image(a).rgb_array(), read_pfm_image(b).rgb_array()), f
        assert (tmp_path / f"f{f:03d}.png").stat().st_size > 100


# ------------------------------------------------------------------ sphere hierarchy (SURVEY §8f-3)
@pytest.mark.parametrize("n_spheres", [1, 3, 37, 1100])
def test_bvh_images_equal_the_linear_scan(n_spheres):
    """accel="bvh" must give the images of the default loop over all shapes (same per-shape tests, same
    tie rule, conservative culling): BIT FOR BIT in fp64 — every renderer, and still equal to the
    oracle's plain loop.  In fp32 the two may differ on a handful of rays, and there the tree is the more
    faithful one: for a ray that starts thousands of units away (the ground near the horizon) the fp32
    discriminant of a far sphere is rounding noise (|o'|^2 ~ 1e8 against a radius of 1), so the scan
    reports phantom hits on spheres the ray passes at a distance; the tree never tests a sphere whose
    box the ray misses.  Bar for fp32: <= 0.1 % of pixels differ."""
    rs = scenes.random_spheres_scene(n_spheres, 2024, 4, 20.0, with_light=True)
    fs = flatten_world(rs.world)
    sc = DeviceScene(fs)
    w, h = (96, 54) if n_spheres > 100 else (64, 36)
    for algo in ("onoff", "flat", "pointlight"):
        for prec in ("f64", "f32"):
            kw = dict(precision=prec, out_f64=(prec == "f64"), aa_pcg=PCG(42, 54))
            a, ha, sa = sc.render(make_params(w, h, rs.camera, algo, 2, **kw), want_hit=True)
            b, hb, sb = sc.render(make_params(w, h, rs.camera, algo, 2, accel="bvh", **kw), want_hit=True)
            assert sa["rays_closest"] == sb["rays_closest"]
            if prec == "f64":
                assert np.array_equal(ha, hb) and np.array_equal(a, b), algo
                assert sa["rays_shadow"] == sb["rays_shadow"]
            else:
                assert (ha != hb).mean() <= 1e-3 and (a != b).any(axis=-1).mean() <= 1e-3, algo
    ref = oracle.render(fs, make_params(w, h, rs.camera, "pointlight", 0, out_f64=True))
    rgb, hit, st = sc.render(make_params(w, h, rs.camera, "pointlight", 0, out_f64=True, accel="bvh"), want_hit=True)
    assert np.array_equal(hit, ref["hit_index"]) and st["rays_shadow"] == ref["rays_shadow"]
    assert np.allclose(rgb, ref["rgb"], rtol=1e-9, atol=1e-12)
    # path tracing: fp64 megakernel bit for bit (same streams, same tree); fp32 kernels within the bar above
    kw = dict(algorithm="pathtracing", samples_per_side=2, num_of_rays=3, max_depth=3, rr_limit=2,
              aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), hit_mode=_abi.RT_HIT_RAY_COUNT)
    a, ca, sa = sc.render(make_params(w, h, rs.camera, variant="mega", precision="f64", out_f64=True, **kw), want_hit=True)
    b, cb, sb = sc.render(make_params(w, h, rs.camera, variant="mega", precision="f64", out_f64=True, accel="bvh", **kw), want_hit=True)
    assert np.array_equal(ca, cb) and np.array_equal(a, b) and sa["rays_closest"] == sb["rays_closest"]
    for variant in ("warp", "mega"):
        a, ca, sa = sc.render(make_params(w, h, rs.camera, variant=variant, **kw), want_hit=True)
        b, cb, sb = sc.render(make_params(w, h, rs.camera, variant=variant, accel="bvh", **kw), want_hit=True)
        assert sb["overflow"] == 0
        assert (ca != cb).mean() <= 2e-3, variant  # the same ray tree, pixel by pixel
        same = ca == cb
        # (the warp kernel adds a pixel's contributions in lane order, which differs between the modes)
        assert np.allclose(a[same], b[same], rtol=2e-5, atol=1e-6) or variant == "mega"
        assert abs(luminosity(a).mean() - luminosity(b).mean()) <= 2e-3 * luminosity(a).mean()


def test_bvh_follows_transform_updates_and_full_size_config5():
    """The hierarchy is rebuilt after rt_scene_update_transforms; BASELINE config 5 at full size
    (3840x2160, 4 spp, 4096 ellipsoids, point light): bvh == linear scan on all 8.3 M pixels."""
    from pytracer_b200.scene import Vec, translation

    rs = scenes.random_spheres_scene(64, 5, 6, 8.0, with_light=True)
    sc = DeviceScene(rs.world)
    p_lin = make_params(80, 45, rs.camera, "flat", 0, precision="f32")
    p_bvh = make_params(80, 45, rs.camera, "flat", 0, precision="f32", accel="bvh")
    assert (sc.render(p_lin)[0] != sc.render(p_bvh)[0]).any(axis=-1).mean() <= 1e-3
    for shape in rs.world.shapes[:40]:
        shape.transformation = translation(Vec(1.5, -2.0, 0.5)) * shape.transformation
    sc.update_from_world(rs.world)
    moved = sc.render(p_bvh)[0]
    assert (moved != sc.render(p_lin)[0]).any(axis=-1).mean() <= 1e-3
    assert np.array_equal(moved, DeviceScene(rs.world).render(p_bvh)[0])

    rs = scenes.random_spheres_scene(4096, 2025, 5, 40.0, with_light=True)
    sc = DeviceScene(rs.world)
    kw = dict(precision="f32", aa_pcg=PCG(42, 54))
    a, ha, sa = sc.render(make_params(3840, 2160, rs.camera, "pointlight", 2, **kw), want_hit=True)
    b, hb, sb = sc.render(make_params(3840, 2160, rs.camera, "pointlight", 2, accel="bvh", **kw), want_hit=True)
    assert sa["rays_closest"] == sb["rays_closest"]
    assert (ha != hb).mean() <= 1e-4 and (a != b).any(axis=-1).mean() <= 1e-3  # fp32: see the test above
    assert sb["kernel_ms"] < sa["kernel_ms"]
    # fp64, the bit-faithful default of this renderer: a window of the same frame, bit for bit
    kw = dict(precision="f64", out_f64=True, aa_pcg=PCG(42, 54))
    a, ha, sa = sc.render(make_params(384, 216, rs.camera, "pointlight", 2, **kw), want_hit=True)
    b, hb, sb = sc.render(make_params(384, 216, rs.camera, "pointlight", 2, accel="bvh", **kw), want_hit=True)
    assert np.array_equal(ha, hb) and np.array_equal(a, b) and sa["rays_shadow"] == sb["rays_shadow"]


def test_every_kernel_at_tiny_sizes():
    """tests/kernel_sweep.py: each kernel / accumulator mode / accel / precision once at tiny sizes, and the
    edges of the work-stack sizing (N = 1, deep trees, N > 32, N > 1024) — finite images, no work-stack
    overflow, warp == mega in the mean (the script is also what one would run under a memory checker)."""
    import runpy, os

    runpy.run_path(os.path.join(os.path.dirname(os.path.abspath(__file__)), "kernel_sweep.py"))


# ------------------------------------------------------------------ one process, several devices (SURVEY §8b/e)
def test_single_process_multi_gpu_image_is_bit_identical():
    """rt_render_multi / CudaRenderer(gpus=n): every visible device traces its interleaved rows from ONE
    process and one call; image, hit index and counters equal the single-device render bit for bit (each pixel
    is computed by exactly one device with the kernel it would run alone).  Needs >= 2 devices."""
    from pytracer_b200 import _native
    from pytracer_b200.device import MultiDeviceScene
    from pytracer_b200.hdrimage import HdrImage
    from pytracer_b200.imagetracer import CudaImageTracer
    from pytracer_b200.render import PathTracer

    n = _native.require_device().rt_device_count()
    if n < 2:
        pytest.skip("one visible device")
    fs, cam = demo_flat()
    one, many = DeviceScene(fs), MultiDeviceScene(fs, n)
    # (path tracing: with >= 32 samples per pixel a warp's task is one pixel and the pixel's fp32 sum is formed
    # in the same order wherever the pixel is traced; with fewer, pixels share a task, the grouping follows the
    # device's own pixel list and the sum order differs: same samples, equal to fp32 rounding)
    cases = [(dict(algorithm="pathtracing", samples_per_side=6, num_of_rays=4, max_depth=3, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54)), True),
             (dict(algorithm="pathtracing", samples_per_side=3, num_of_rays=4, max_depth=3, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54)), False),
             (dict(algorithm="pointlight", samples_per_side=2, aa_pcg=PCG(42, 54)), True),
             (dict(algorithm="flat", samples_per_side=0, out_f64=True), True)]
    for kw, exact in cases:
        for w, h in ((203, 117), (64, n - 1)):  # odd sizes; fewer rows than devices
            a, ha, sa = one.render(make_params(w, h, cam, **kw), want_hit=True)
            b, hb, sb = many.render(make_params(w, h, cam, **kw), want_hit=True)
            assert np.array_equal(ha, hb), (kw["algorithm"], w, h)
            assert np.array_equal(a, b) if exact else np.allclose(a, b, rtol=1e-5, atol=1e-7), (kw["algorithm"], w, h)
            assert (sa["rays_closest"], sa["rays_shadow"], sa["samples"]) == (sb["rays_closest"], sb["rays_shadow"], sb["samples"])
    with pytest.raises(Exception):  # the call splits the image itself
        many.render(make_params(64, 48, cam, "flat", 0, part_mode=_abi.RT_PART_ROWS, part_rank=0, part_count=2))
    # through the public classes
    world, camera = scenes.demo_scene()
    imgs = []
    for gpus in (1, n):
        image = HdrImage(160, 120)
        CudaImageTracer(image, camera, samples_per_side=6, pcg=PCG(42, 54)).fire_all_rays(
            PathTracer(world, pcg=PCG(45, 54), num_of_rays=5, max_depth=3, gpus=gpus))
        imgs.append(image.rgb_array().copy())
    assert np.array_equal(imgs[0], imgs[1])
    one.close(); many.close()


def test_render_command_with_gpus_writes_the_same_file(tmp_path):
    """`render --gpus N` (all devices from this process): the PFM equals the single-device file byte for byte."""
    from click.testing import CliRunner

    from pytracer_b200 import _native
    from pytracer_b200.main import cli

    n = _native.require_device().rt_device_count()
    if n < 2:
        pytest.skip("one visible device")
    scene_file = tmp_path / "demo.txt"
    scene_file.write_text(DEMO_TEXT)
    files = []
    for gpus in (1, n):
        pfm = tmp_path / f"g{gpus}.pfm"
        res = CliRunner().invoke(cli, ["render", "--width", "200", "--height", "150", "--algorithm", "pointlight", "--samples-per-pixel", "4",
                                       "--gpus", str(gpus), "--pfm-output", str(pfm), "--png-output", str(tmp_path / f"g{gpus}.png"),
                                       "--parser", "builtin", str(scene_file)])
        assert res.exit_code == 0, res.output
        files.append(pfm.read_bytes())
    assert files[0] == files[1]
