"""Pins the CPU oracle (oracle/pt_oracle.c) to the reference: every comparison is against an output
of the unmodified Python reference stored under tests/golden/, and every comparison is BIT-EXACT
(images as fp64 arrays, hit indices, ray counts, final PCG states)."""
import numpy as np
import pytest

from oracle import oracle
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG
from util import c1_params, demo_flat, golden, scene2_flat, sha256_of


def test_pcg_known_answers():
    # tests/test_all.py:872-887
    state, inc = oracle.pcg_seed(42, 54)
    assert (state, inc) == (1753877967969059832, 109)
    draws, _ = oracle.pcg_draw(state, inc, 6)
    assert draws.tolist() == [2707161783, 2068313097, 3122475824, 2211639955, 3215226955, 3421331566]


def test_c1_pathtracing_image_is_bit_exact():
    fs, cam = demo_flat()
    g = golden("demo_c1_pathtracing_160x120.npz")
    r = oracle.render(fs, c1_params(cam))
    assert np.array_equal(r["rgb"], g["rgb"])
    assert r["rays_closest"] == int(g["rays_closest"]) == 393440
    assert r["pt_state"] == int(g["pt_state_end"])
    assert r["aa_state"] == int(g["aa_state_end"])


@pytest.mark.parametrize("algo", ["onoff", "flat", "pointlight"])
@pytest.mark.parametrize("s,size", [(0, (160, 120)), (2, (64, 48))])
def test_deterministic_renderers_bit_exact(algo, s, size):
    fs, cam = demo_flat()
    g = golden("demo_deterministic.npz")
    r = oracle.render(fs, make_params(size[0], size[1], cam, algo, s, aa_pcg=PCG(42, 54)))
    assert np.array_equal(r["rgb"], g[f"{algo}_s{s}_rgb"])
    assert np.array_equal(r["hit_index"], g[f"hit_s{s}"])
    assert r["rays_closest"] == int(g[f"{algo}_s{s}_rays_closest"])
    assert r["rays_shadow"] == int(g[f"{algo}_s{s}_rays_shadow"])
    assert r["aa_state"] == int(g[f"{algo}_s{s}_aa_state_end"])


def test_roulette_inside_the_tree_bit_exact():
    fs, cam = demo_flat()
    g = golden("demo_pt_small.npz")
    p = make_params(40, 30, cam, "pathtracing", 2, num_of_rays=3, max_depth=5, rr_limit=2,
                    aa_pcg=PCG(7, 11), pt_pcg=PCG(99, 3), background=(0.05, 0.02, 0.01))
    r = oracle.render(fs, p)
    assert np.array_equal(r["rgb"], g["rgb"])
    assert r["rays_closest"] == int(g["rays_closest"])
    assert r["pt_state"] == int(g["pt_state_end"])


@pytest.mark.parametrize("tag", ["persp", "ortho"])
def test_scene2_all_renderers_bit_exact(tag):
    fs, cam_p, cam_o = scene2_flat()
    cam = cam_p if tag == "persp" else cam_o
    g = golden("scene2.npz")
    bg = (0.02, 0.03, 0.04)
    for algo in ("onoff", "flat", "pointlight"):
        r = oracle.render(fs, make_params(96, 64, cam, algo, 0, background=bg))
        assert np.array_equal(r["rgb"], g[f"{tag}_{algo}_rgb"]), algo
        assert np.array_equal(r["hit_index"], g[f"{tag}_hit"])
        assert r["rays_shadow"] == int(g[f"{tag}_{algo}_rays_shadow"])
    p = make_params(48, 32, cam, "pathtracing", 2, num_of_rays=4, max_depth=4, rr_limit=2,
                    aa_pcg=PCG(5, 9), pt_pcg=PCG(123, 77), background=bg)
    r = oracle.render(fs, p)
    assert np.array_equal(r["rgb"], g[f"{tag}_pt_rgb"])
    assert r["rays_closest"] == int(g[f"{tag}_pt_rays_closest"])
    assert r["pt_state"] == int(g[f"{tag}_pt_pt_state_end"])


def test_per_function_known_answers_bit_exact():
    fs, cam_p, cam_o = scene2_flat()
    k = golden("scene2_kat.npz")
    hits = oracle.intersect(fs, k["rays"])
    for h, ref in zip(hits, k["hits"]):
        assert h.shape == int(ref[0])
        if h.shape >= 0:
            got = [h.t, *h.world_point, *h.normal, *h.uv]
            assert got == ref[1:10].tolist()
    assert np.array_equal(oracle.is_point_visible(fs, k["pairs"]), k["visible"].astype(bool))
    st, inc = oracle.pcg_seed(17, 5)
    out, end = oracle.scatter(fs, 0, k["scatter_in"], st, inc)  # material 0 = diffuse image pigment
    assert np.array_equal(out, k["scatter_diffuse"]) and end == int(k["scatter_diffuse_state_end"])
    out, end = oracle.scatter(fs, 1, k["scatter_in"], st, inc)  # material 1 = specular
    assert np.array_equal(out, k["scatter_specular"]) and end == int(k["scatter_specular_state_end"])
    assert np.array_equal(oracle.onb(k["onb_in"]), k["onb_out"])


def test_pigments_and_cameras_bit_exact():
    fs, cam_p, cam_o = scene2_flat()
    k = golden("scene2_kat.npz")
    mats = fs.materials
    # pigments in the order make_golden.py sampled them: image (shape 0), checkered (shape 3),
    # uniform (shape 1), checkered emitter (shape 5)
    idx = [mats[fs.shape_material[0]].brdf_pigment, mats[fs.shape_material[3]].brdf_pigment,
           mats[fs.shape_material[1]].brdf_pigment, mats[fs.shape_material[5]].emitted_pigment]
    for j, pig in enumerate(idx):
        assert np.array_equal(oracle.pigment_color(fs, pig, k["uv"]), k[f"pigment{j}"])


def test_renderer_calls_on_explicit_rays_bit_exact():
    fs, cam_p, _ = scene2_flat()
    k = golden("scene2_kat.npz")
    bg = (0.02, 0.03, 0.04)
    for algo in ("onoff", "flat", "pointlight"):
        p = make_params(1, 1, cam_p, algo, background=bg)
        out, _, _ = oracle.trace_rays(fs, p, k["call_rays"])
        assert np.array_equal(out, k[f"call_{algo}"]), algo
    pcg = PCG(31, 41)
    p = make_params(1, 1, cam_p, "pathtracing", num_of_rays=2, max_depth=4, rr_limit=1, background=bg, pt_pcg=pcg)
    depth = np.arange(300, dtype=np.int32) % 3
    out, (state, _), _ = oracle.trace_rays(fs, p, k["call_rays"], depth)
    assert np.array_equal(out, k["call_pathtracing"])
    assert state == int(k["call_pathtracing_state_end"])


def test_furnace_matches_the_reference_run():
    # tests/test_all.py:1014-1051, values produced by the reference's PathTracer
    from pytracer_b200 import Color, DiffuseBRDF, Material, Sphere, UniformPigment, World
    from pytracer_b200.flatten import flatten_world
    from pytracer_b200.scene import PerspectiveCamera

    a = golden("analytic.npz")
    for i, (emitted, refl, r, g, b, expected) in enumerate(a["furnace"]):
        world = World()
        world.add_shape(Sphere(material=Material(DiffuseBRDF(UniformPigment(Color(refl, refl, refl))),
                                                 UniformPigment(Color(emitted, emitted, emitted)))))
        fs = flatten_world(world)
        p = make_params(1, 1, PerspectiveCamera(), "pathtracing", num_of_rays=1, max_depth=100, rr_limit=101)
        inc = PCG().inc
        out, (state, _), _ = oracle.trace_rays(fs, p, np.array([[0, 0, 0, 1, 0, 0, 1e-5, np.inf]]),
                                               pcg_state_inc=(int(a[f"furnace_state0_{i}"]), inc))
        assert out[0].tolist() == [r, g, b]
        assert state == int(a[f"furnace_state1_{i}"])
        assert abs(out[0][0] - expected) < 1e-3 * expected + 1e-3


def test_1080p_config2_bit_exact():
    fs, cam = demo_flat()
    g = golden("demo_1080p.npz")
    r = oracle.render(fs, make_params(1920, 1080, cam, "flat", 0))
    assert np.array_equal(r["hit_index"], g["hit"].astype(np.int32))
    assert np.array_equal(r["rgb"].astype(np.float32), g["flat_rgb_f32"])
    counts = np.bincount(r["hit_index"].ravel() + 1, minlength=4)
    assert counts.tolist() == [484487, 518387, 1002874, 67852]  # BASELINE.md golden anchors
    r = oracle.render(fs, make_params(1920, 1080, cam, "pointlight", 0))
    assert sha256_of(r["rgb"].astype(np.float32)) == str(g["pointlight_rgb_f32_sha256"])
    assert [r["rays_closest"], r["rays_shadow"]] == g["pointlight_rays"].tolist() == [2073600, 1589113]


# ------------------------------------------------------------------ tone mapping (SURVEY §8f-2)
def tonemap_cases():
    g = golden("tonemap.npz")
    for i in range(int(g["n_cases"])):
        factor, lum, gamma = (float(x) for x in g[f"case{i}_params"])
        yield i, g[f"img_{str(g[f'case{i}_image'])}"], factor, (None if np.isnan(lum) else lum), gamma, g


def test_tonemap_oracle_matches_the_reference():
    from oracle import tonemap_oracle as tm

    for i, img, factor, lum, gamma, g in tonemap_cases():
        avg = tm.average_luminosity(img)
        assert avg == float(g[f"case{i}_avg"])  # same logs added in the same order
        used, hdr, ldr = tm.tone_map(img, factor, lum, gamma)
        assert np.allclose(hdr, g[f"case{i}_hdr"], rtol=1e-15, atol=0)
        assert np.array_equal(ldr, g[f"case{i}_ldr"])  # bit-exact bytes of the reference's PNG
    # tests/test_all.py:239-268
    kat = np.array([[[5.0, 10.0, 15.0], [500.0, 1000.0, 1500.0]]])
    assert abs(tm.average_luminosity(kat, delta=0.0) - 100.0) < 1e-9
    assert abs(tm.average_luminosity(kat, delta=0.0) - float(golden("tonemap.npz")["kat_avg_delta0"])) < 1e-12
    out = tm.normalize_and_clamp(kat, factor=1000.0, luminosity_value=100.0)
    assert np.allclose(out / (1 - out), [[0.5e2, 1.0e2, 1.5e2], [0.5e4, 1.0e4, 1.5e4]])
    assert (out >= 0).all() and (out <= 1).all()


def test_config4_oracle_fixture_is_reproducible():
    """tests/golden/c4_oracle_64x36.npz (the statistics the full-size config-4 GPU test is held against) is
    what the oracle computes: the rows of run 0 that thread 0 of oracle.render_threaded(…, 8) owns are
    re-rendered here (its first two rows, 0 and 8, in its sequential stream order; 1 026 shapes: ~10 s)."""
    from pytracer_b200 import _abi, scenes
    from pytracer_b200.flatten import flatten_world
    from pytracer_b200.pcg import PCG

    fix = golden("c4_oracle_64x36.npz")
    threads, spp = int(fix["threads"]), int(fix["spp_per_run"])
    assert fix["runs"].shape == (16, 36, 64, 3) and spp == 16
    rs = scenes.random_spheres_scene(1024, 2024, 4, 20.0)
    fs = flatten_world(rs.world)
    p = make_params(64, 36, rs.camera, algorithm="pathtracing", samples_per_side=4, num_of_rays=10, max_depth=3, rr_limit=3,
                    aa_pcg=PCG(1000, 7), pt_pcg=PCG(2000, 9))
    q = _abi.rt_render_params.from_buffer_copy(bytes(p))   # thread 0's streams, as render_threaded derives them
    aa, pt = PCG(p.aa_state & 0xFFFFFFFF, 1000), PCG(p.pt_state & 0xFFFFFFFF, 2000)
    q.aa_state, q.aa_inc, q.pt_state, q.pt_inc = aa.state, aa.inc, pt.state, pt.inc
    r = oracle.render(fs, q, 0, threads + 1, want_hit=False, row_step=threads)
    rows = [0, threads]
    assert np.array_equal(r["rgb"][rows].astype(np.float32), fix["runs"][0][rows])
    assert abs(float(fix["rays_per_sample"]) - 127.0) < 0.5
