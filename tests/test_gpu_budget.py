"""rt_render_adaptive_budget / fire_all_rays_adaptive(mean_samples_per_pixel=...) on the device: one pass equals
`render`, the first selection is exactly the host's (e descending, pixel index ascending), a cut inside a group of
exactly tied errors is resolved by pixel index, the passes replay on the host from single-pass renders, the budget is
accounted for, and the accel, estimator, oracle and command-line paths agree."""
import numpy as np
import pytest

from oracle import oracle
from pytracer_b200 import scenes
from pytracer_b200.device import DeviceScene
from pytracer_b200.flatten import flatten_world
from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.imagetracer import CudaImageTracer
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG, lcg_advance
from pytracer_b200.render import PathTracer
from pytracer_b200.scene_text import parse_scene_text
from test_adaptive_cpu import DEMO_TXT
from test_budget_cpu import pass_size, select_pixels
from util import assert_luminance_agreement, assert_mc_agreement, demo_flat

pytestmark = pytest.mark.gpu

PT = dict(algorithm="pathtracing", num_of_rays=10, max_depth=3, rr_limit=3)


def _params(w, h, cam, S, pas=0, **kw):
    """Parameters of pass `pas`: the jitter state advanced by pas * 2 * W * H * S^2 draws, the path-tracing state by
    pas steps (pas = 0: the parameters of the whole call)."""
    p = make_params(w, h, cam, samples_per_side=S, aa_pcg=PCG(11, 3), pt_pcg=PCG(77, 5), **dict(PT, **kw))
    p.aa_state = lcg_advance(p.aa_state, p.aa_inc, pas * 2 * w * h * S * S)
    p.pt_state = lcg_advance(p.pt_state, p.pt_inc, pas)
    return p


def _pass0_error(mean, err, floor=1e-2):
    """e of every pixel after one pass, exactly as the device forms it in fp32 (P = 1: mean and SE are the sums)."""
    return (err / np.maximum(mean, np.float32(floor))).max(-1)


def _flagged_twice(samples, S2):
    return np.flatnonzero((samples == 2 * S2).ravel())


def test_one_pass_budget_equals_render():
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    S, W, H = 4, 160, 120
    p = _params(W, H, cam, S)
    rgb, _, st = sc.render(p)
    mean, err, samples, bst = sc.render_budget(p, W * H * S * S, 8)
    assert np.array_equal(mean, rgb)
    assert bst["passes"] == 1 and bst["pixels_in_pass"] == [W * H] and (samples == S * S).all()
    assert (bst["rays_closest"], bst["rays_shadow"], bst["samples"]) == (st["rays_closest"], st["rays_shadow"], st["samples"])
    assert bst["overflow"] == 0 and np.isfinite(err).all()


@pytest.mark.parametrize("target", [0.0, 0.05])
def test_first_selection_is_exact(target):
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    S, W, H = 4, 160, 120
    S2, n = S * S, W * H
    p = _params(W, H, cam, S)
    m0, e0, _, _ = sc.render_adaptive(p, 0.0, 1)
    e = _pass0_error(m0, e0)
    C = int((e > np.float32(target)).sum())
    print(f"target {target}: {C} candidates of {n}")
    assert 0 < C < n
    for K in (1, 7, 100, 2048 + 5, C - 1, C, C + 500):
        _, _, samples, st = sc.render_budget(p, (n + K) * S2, 2, target)
        want = select_pixels(e, target, min(C, K))
        got = _flagged_twice(samples, S2)
        assert np.array_equal(got, want), (K, len(got), len(want))
        assert st["pixels_in_pass"] == [n, min(C, K)] and st["samples"] == (n + min(C, K)) * S2


TIES_TXT = """
material emitter(diffuse(uniform(<0, 0, 0>)), {pigment})
plane(emitter, translation([2, 0, 0]) * rotation_y(90))
camera(perspective, identity, 1.0, 1.0)
"""


def _emitter_scene(pigment):
    parsed = parse_scene_text(TIES_TXT.format(pigment=pigment))
    return DeviceScene(flatten_world(parsed.world)), parsed.camera


def test_a_cut_inside_a_tie_group_is_resolved_by_pixel_index():
    """An emissive plane checkered in 0.5 and 0.25, seen directly (max_depth 0): every sample is one of two dyadic
    values, so every sum is exact, and e of a pixel depends only on how many of its 16 samples saw each colour."""
    sc, cam = _emitter_scene("checkered(<0.5, 0.5, 0.5>, <0.25, 0.25, 0.25>, 32)")
    S, W, H = 4, 128, 96
    S2, n = S * S, W * H
    p = make_params(W, H, cam, samples_per_side=S, aa_pcg=PCG(5, 6), pt_pcg=PCG(7, 8), algorithm="pathtracing",
                    num_of_rays=1, max_depth=0, rr_limit=3)
    m0, e0, _, _ = sc.render_adaptive(p, 0.0, 1)
    assert np.isin(m0, np.arange(17, dtype=np.float32) / np.float32(64) + np.float32(0.25)).all()  # 0.25 + a / 64, exact
    e = _pass0_error(m0, e0).ravel()
    values, counts = np.unique(e[e > 0], return_counts=True)
    print(f"{int((e > 0).sum())} candidates in {len(values)} groups of equal e: {counts[::-1].tolist()}")
    assert len(values) <= 15 and counts.max() >= 500
    # cut the largest group in its middle
    g = int(np.argmax(counts))
    above = int(counts[g + 1:].sum())
    for K in (above + 1, above + counts[g] // 2, above + counts[g] - 1):
        order = np.sort(e)[::-1]
        assert order[K - 1] == order[K] == values[g]  # the K-th and the (K+1)-th pixel tie
        mean, _, samples, st = sc.render_budget(p, (n + K) * S2, 2)
        got = _flagged_twice(samples, S2)
        want = select_pixels(e, 0.0, K)
        assert np.array_equal(got, want), K
        in_group = np.flatnonzero(e == values[g])
        taken = np.intersect1d(got, in_group)
        assert np.array_equal(taken, in_group[:K - above])  # the lowest pixel indices of the group
    # a uniform emitter has no error: no candidate, one pass whatever the budget
    sc, cam = _emitter_scene("uniform(<0.5, 0.25, 0.5>)")
    mean, err, samples, st = sc.render_budget(p, 10 * n * S2, 8)
    assert st["passes"] == 1 and (samples == S2).all() and (err == 0).all() and st["samples"] == n * S2


def _replay_budget(means, errs, budget, max_passes, target, floor, S2, band=1e-6):
    """Host replica of rt_render_adaptive_budget from what every pass gives each pixel ([K][H][W][3] mean and SE of
    single-pass renders).  Sums as in tests/util.py replay_adaptive: the mean in fp32 in pass order (exact), the SE^2
    in fp64 from the observable SE (approximate where P >= 2, exact in fp32 where P = 1).  `ambiguous` counts the
    decisions an approximate e came within a relative `band` of: the target, or the error at the cut.
    The band: SE_p = RN(sqrt(SE_p^2)) squares back within 2^-23 of the device's SE_p^2, and the device's fp32 sum of
    P terms adds at most (P - 1) 2^-24, so sqrt(sum) is off by (P + 1) 2^-25; the device rounds the square root and two
    divisions (3 x 2^-24).  For P <= 8 that is 4.5e-7 of e, and twice that at a cut between two such values."""
    K_, H, W, _ = means.shape
    m = means.reshape(K_, -1, 3).astype(np.float32)
    v = errs.reshape(K_, -1, 3).astype(np.float64) ** 2
    n = H * W
    sum_m, sum_v = m[0].copy(), v[0].copy()
    P = np.ones(n, dtype=np.int32)
    t, fl = float(np.float32(target)), np.float32(floor)
    spent, pixels_in_pass, cands, ambiguous = n * S2, [n], [], 0
    for p in range(max_passes - 1):
        mean = sum_m / P[:, None].astype(np.float32)
        e = (np.sqrt(sum_v) / P[:, None] / np.maximum(mean, fl)).max(-1)
        exact = P == 1
        e[exact] = e[exact].astype(np.float32)
        cand = np.flatnonzero(e > t)
        if t > 0:
            ambiguous += int((~exact & (np.abs(e / t - 1.0) < band)).sum())
        C, Q = len(cand), (budget - spent) // S2
        cands.append(C)
        K = pass_size(C, Q, max_passes - 1 - p)
        if K == 0:
            break
        order = cand[np.lexsort((cand, -e[cand]))]
        if K < C:
            a, b = order[K - 1], order[K]
            if not (exact[a] and exact[b]) and e[a] - e[b] <= band * e[a]:
                ambiguous += 1
        sel = np.sort(order[:K])
        sum_m[sel] = sum_m[sel] + m[p + 1][sel]
        sum_v[sel] += v[p + 1][sel]
        P[sel] += 1
        spent += K * S2
        pixels_in_pass.append(K)
    return dict(mean=(sum_m / P[:, None].astype(np.float32)).reshape(H, W, 3), P=P.reshape(H, W), spent=spent,
                pixels_in_pass=pixels_in_pass, candidates=cands, ambiguous=ambiguous)


@pytest.mark.parametrize("mean_spp, max_passes, target", [(96, 4, 0.0), (160, 8, 0.0), (128, 6, 0.03), (400, 4, 0.05), (80, 2, 0.0)])
def test_passes_replay_on_the_host_and_the_budget_adds_up(mean_spp, max_passes, target):
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    S, W, H = 8, 160, 120
    S2, n = S * S, W * H
    assert max_passes <= 8  # (the band of _replay_budget)
    budget = mean_spp * n
    means, errs = [], []
    for pas in range(max_passes):
        mp, ep, _, _ = sc.render_adaptive(_params(W, H, cam, S, pas), 0.0, 1)
        means.append(mp)
        errs.append(ep)
    # a target that no approximate e of the replay lies within the band of (chosen on the host, before the device call)
    for t in ([target] if target == 0 else [target * f for f in (1.0, 0.97, 1.03, 0.94, 1.06)]):
        r = _replay_budget(np.stack(means), np.stack(errs), budget, max_passes, t, 1e-2, S2)
        if r["ambiguous"] == 0:
            target = t
            break
    mean, err, samples, st = sc.render_budget(_params(W, H, cam, S), budget, max_passes, target)
    print(f"mean {mean_spp}, M {max_passes}, target {target}: pixels per pass {st['pixels_in_pass']} (host "
          f"{r['pixels_in_pass']}), candidates {r['candidates']}, {st['samples']} of {budget} samples, "
          f"{r['ambiguous']} ambiguous decisions")
    assert r["ambiguous"] == 0  # so that the comparison below means something
    assert st["pixels_in_pass"] == r["pixels_in_pass"] and st["passes"] == len(r["pixels_in_pass"])
    assert np.array_equal(samples // S2, r["P"]) and (samples % S2 == 0).all()
    assert np.array_equal(mean, r["mean"])  # one pixel per task at S^2 = 64: the same sums in the same order
    # the budget: spent = the samples every pixel reports, at most B; what is left is less than one pixel pass unless
    # the candidates ran out or the pass limit came first
    assert st["samples"] == int(samples.sum()) == r["spent"] <= budget and st["overflow"] == 0
    assert budget - st["samples"] < S2 or r["candidates"][-1] == 0 or st["passes"] == max_passes
    spent = n * S2
    for p, K in enumerate(st["pixels_in_pass"][1:]):
        C, Q = r["candidates"][p], (budget - spent) // S2
        assert K >= min(-(-C // 2), Q), (p, K, C, Q)  # at least half of the candidates where the budget allows
        spent += K * S2
    assert (samples <= max_passes * S2).all()


def test_deterministic_and_leaves_the_streams_where_plain_renders_do():
    world, camera = scenes.demo_scene()

    def run():
        tracer = CudaImageTracer(HdrImage(160, 120), camera, samples_per_side=4, pcg=PCG(42, 54))
        renderer = PathTracer(world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3)
        res = tracer.fire_all_rays_adaptive(renderer, mean_samples_per_pixel=40, max_samples_per_pixel=160)
        return tracer, renderer, res

    tracer, renderer, res = run()
    again = run()
    assert np.array_equal(tracer.image.rgb_array(), again[0].image.rgb_array())
    assert np.array_equal(res.error, again[2].error) and np.array_equal(res.samples, again[2].samples)
    assert res.passes >= 3 and res.stats["sample_budget"] == 40 * 160 * 120 and res.stats["samples"] <= 40 * 160 * 120
    plain_t = CudaImageTracer(HdrImage(160, 120), camera, samples_per_side=4, pcg=PCG(42, 54))
    plain_r = PathTracer(world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3)
    for _ in range(res.passes):
        plain_t.fire_all_rays(plain_r)
    assert (tracer.pcg.state, renderer.pcg.state) == (plain_t.pcg.state, plain_r.pcg.state)


def test_the_hierarchy_path_and_the_paired_estimator():
    """37 random spheres with accel="bvh" (k_pt_warp_bvh): one pass equals `render` with the hierarchy bit for bit, and
    the first selection is exactly the host's from that pass.  (The fp32 warp kernels add a pixel's contributions in
    lane order, which differs between accel="bvh" and "none", so the two images agree only to rounding:
    tests/test_gpu_parity.py test_bvh_images_equal_the_linear_scan.)"""
    rs = scenes.random_spheres_scene(37)
    sc = DeviceScene(flatten_world(rs.world))
    kw = dict(num_of_rays=4, max_depth=3, rr_limit=2)
    S, W, H = 4, 160, 120
    S2, n = S * S, W * H
    B = 48 * n
    for accel in ("bvh", "none"):
        p = _params(W, H, rs.camera, S, accel=accel, **kw)
        rgb, _, st = sc.render(p)
        mean, _, samples, bst = sc.render_budget(p, n * S2, 8)
        assert np.array_equal(mean, rgb) and bst["passes"] == 1 and bst["rays_closest"] == st["rays_closest"], accel
        m0, e0, _, _ = sc.render_adaptive(p, 0.0, 1)
        e = _pass0_error(m0, e0)
        C = int((e > 0).sum())
        for K in (333, C // 2 + 1):
            _, _, samples, bst = sc.render_budget(p, (n + K) * S2, 2)
            assert np.array_equal(_flagged_twice(samples, S2), select_pixels(e, 0.0, min(C, K))), (accel, K)
        mean, err, samples, bst = sc.render_budget(p, B, 8)
        print(f"spheres37 {accel}: pixels per pass {bst['pixels_in_pass']}, {bst['samples']} of {B} samples")
        assert bst["passes"] >= 3 and bst["samples"] == int(samples.sum()) <= B and bst["overflow"] == 0
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    mean, err, samples, st = sc.render_budget(_params(W, H, cam, S), B, 8, estimator="paired")
    print(f"paired: pixels per pass {st['pixels_in_pass']}, {st['samples']} of {B} samples")
    assert st["passes"] >= 3 and st["samples"] == int(samples.sum()) <= B and np.isfinite(err).all()
    assert B - st["samples"] < 16 or st["passes"] == 8


def test_budget_image_agrees_with_the_reference_estimator():
    import os

    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    p = make_params(160, 120, cam, samples_per_side=4, aa_pcg=PCG(11, 3), pt_pcg=PCG(77, 5), **PT)
    mean, err, samples, st = sc.render_budget(p, 64 * 160 * 120, 64)
    print(f"budget demo.txt: passes {st['passes']}, pixels per pass {st['pixels_in_pass']}, {st['samples']} samples "
          f"({st['samples'] / samples.size:.1f} per pixel), {st['kernel_ms']:.2f} ms")
    assert st["samples"] == int(samples.sum()) <= 64 * 160 * 120 and (samples >= 16).all() and (samples <= 1024).all()
    threads = max(1, min(32, os.cpu_count() or 1))
    ref = np.stack([oracle.render_threaded(fs, make_params(160, 120, cam, samples_per_side=4, aa_pcg=PCG(1000 + k, 7),
                                                           pt_pcg=PCG(2000 + k, 9), **PT), threads)["rgb"].copy()
                    for k in range(24)])
    gpu = mean.astype(np.float64)
    assert_luminance_agreement(gpu, ref, what="budget demo.txt 160x120")
    assert_mc_agreement(gpu, ref, samples_ratio=(24 * 16) / samples[..., None].astype(np.float64), n_ref=24 * 16,
                        what="budget demo.txt 160x120")


def test_render_command_writes_the_in_process_image(tmp_path):
    from click.testing import CliRunner

    from pytracer_b200.hdrimage import read_pfm_image
    from pytracer_b200.main import cli

    scene = tmp_path / "demo.txt"
    scene.write_text(DEMO_TXT)
    out = {k: tmp_path / f"{k}" for k in ("img.pfm", "img.png", "err.pfm")}
    result = CliRunner().invoke(cli, ["render", "--width", "96", "--height", "72", "--samples-per-pixel", "16",
                                      "--mean-samples-per-pixel", "40", "--max-samples-per-pixel", "128",
                                      "--error-estimator", "paired", "--pfm-output", str(out["img.pfm"]),
                                      "--png-output", str(out["img.png"]), "--error-output", str(out["err.pfm"]), str(scene)])
    print(result.output)
    assert result.exit_code == 0, result.output
    assert all(p.exists() and p.stat().st_size > 0 for p in out.values())
    assert f"budget {40 * 96 * 72} samples" in result.output
    parsed = parse_scene_text(DEMO_TXT)
    image = HdrImage(96, 72)
    tracer = CudaImageTracer(image, parsed.camera, samples_per_side=4)
    res = tracer.fire_all_rays_adaptive(PathTracer(parsed.world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3),
                                        mean_samples_per_pixel=40, max_samples_per_pixel=128, error_estimator="paired")
    with open(tmp_path / "inproc.pfm", "wb") as f:
        image.write_pfm(f)
    assert (tmp_path / "inproc.pfm").read_bytes() == out["img.pfm"].read_bytes()
    assert res.passes >= 2
    with open(out["err.pfm"], "rb") as f:
        err = read_pfm_image(f)
    assert np.allclose(err.rgb_array(), res.error)
