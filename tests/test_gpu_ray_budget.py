"""rt_render_adaptive_rays / fire_all_rays_adaptive(mean_rays_per_pixel=...) on the device: one pass equals `render` and
its per-pixel rays equal `render`'s RT_HIT_RAY_COUNT side image in every kernel; the first selection is exactly the host
replica's prefix (tests/test_ray_budget_cpu.py) from the pass-0 mean, SE and ray map; a cut inside a group of exactly
tied keys is resolved by pixel index; multi-pass runs replay on the host bit for bit with the budget's guarantees; the
result is deterministic, leaves the streams where plain renders do, and the command line writes the in-process image."""
import numpy as np
import pytest

from pytracer_b200 import _abi, scenes
from pytracer_b200.device import DeviceScene
from pytracer_b200.flatten import flatten_world
from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.imagetracer import CudaImageTracer
from pytracer_b200.pcg import PCG
from pytracer_b200.render import PathTracer
from pytracer_b200.scene_text import parse_scene_text
from test_adaptive_cpu import DEMO_TXT
from test_budget_cpu import select_pixels
from test_gpu_budget import _emitter_scene, _flagged_twice, _params, _pass0_error
from test_ray_budget_cpu import FLT_MIN, predicted_cost, ray_key, select_prefix, spend_target
from util import demo_flat

pytestmark = pytest.mark.gpu

SPHERES = dict(num_of_rays=4, max_depth=3, rr_limit=2)


def _spheres():
    rs = scenes.random_spheres_scene(37)
    return DeviceScene(flatten_world(rs.world)), rs.camera


@pytest.mark.parametrize("scene, accel, S", [("demo", "none", 8), ("demo", "none", 4), ("demo", "none", 2),
                                             ("spheres", "none", 8), ("spheres", "none", 4), ("spheres", "bvh", 4),
                                             ("spheres", "bvh", 2)])
def test_one_pass_equals_render_and_its_ray_counts(scene, accel, S):
    """S = 8: one-pixel tasks; S = 4 and 2: multi-pixel tasks; demo.txt runs the SMALL kernel, 37 spheres the large-scene
    kernel (accel "none") and k_pt_warp_bvh (accel "bvh")."""
    if scene == "demo":
        fs, cam = demo_flat()
        sc, kw = DeviceScene(fs), {}
    else:
        (sc, cam), kw = _spheres(), SPHERES
    W, H = 160, 120
    p = _params(W, H, cam, S, accel=accel, **kw)
    rgb, _, st = sc.render(p)
    _, counts, cst = sc.render(_params(W, H, cam, S, accel=accel, hit_mode=_abi.RT_HIT_RAY_COUNT, **kw), want_hit=True)
    mean, err, samples, rays, rst = sc.render_rays(p, 0, 1)
    assert np.array_equal(mean, rgb) and (samples == S * S).all() and np.isfinite(err).all()
    assert rays.dtype == np.int64 and np.array_equal(rays, counts.astype(np.int64))
    assert int(rays.sum()) == rst["rays_closest"] == st["rays_closest"] == cst["rays_closest"]
    assert rst["passes"] == 1 and rst["overflow"] == 0 and (rays >= S * S).all()


@pytest.mark.parametrize("scene", ["demo", "spheres-bvh"])
@pytest.mark.parametrize("target", [0.0, 0.05])
def test_first_selection_is_the_host_prefix(scene, target):
    if scene == "demo":
        fs, cam = demo_flat()
        sc = DeviceScene(fs)
        p = _params(160, 120, cam, 4)
    else:
        sc, cam = _spheres()
        p = _params(160, 120, cam, 4, accel="bvh", **SPHERES)
    S2, n = 16, 160 * 120
    m0, e0, _, r0, st0 = sc.render_rays(p, 0, 1)
    rays0 = st0["rays_closest"]
    e = _pass0_error(m0, e0).ravel()
    w = predicted_cost(r0.ravel(), 1)
    key = ray_key(e, 1, w, target)
    W_c = int(w[key > 0].sum())
    print(f"{scene}, target {target}: {int((key > 0).sum())} candidates of {n}, W_c {W_c}, pass 0 {rays0} rays")
    assert 0 < (key > 0).sum() < n
    for extra in (1, W_c // 7, W_c // 2 + 3, W_c - 1, W_c + 1000, -5):
        R = rays0 + extra
        _, _, samples, rays, st = sc.render_rays(p, R, 2, target)
        want = select_prefix(key, w, spend_target(R - rays0, W_c, 1))  # r = 1 after pass 0 of two
        got = _flagged_twice(samples, S2)
        assert np.array_equal(got, want), (extra, len(got), len(want))
        assert st["pixels_in_pass"] == ([n, len(want)] if len(want) else [n]) and st["passes"] == (2 if len(want) else 1)
        assert int(w[want].sum()) <= max(R - rays0, 0)
        assert st["rays_closest"] == int(rays.sum()) and np.array_equal(np.delete(rays.ravel(), want), np.delete(r0.ravel(), want))


def test_a_cut_inside_a_tie_group_is_resolved_by_pixel_index():
    """The emissive checkered plane of test_gpu_budget.py seen directly (max_depth 0, one ray per sample): every pixel
    costs 16 rays a pass, so equal e give exactly equal keys, and T = 16 K cuts after K pixels."""
    from pytracer_b200.params import make_params

    sc, cam = _emitter_scene("checkered(<0.5, 0.5, 0.5>, <0.25, 0.25, 0.25>, 32)")
    S, W, H = 4, 128, 96
    S2, n = S * S, W * H
    p = make_params(W, H, cam, samples_per_side=S, aa_pcg=PCG(5, 6), pt_pcg=PCG(7, 8), algorithm="pathtracing",
                    num_of_rays=1, max_depth=0, rr_limit=3)
    m0, e0, _, r0, st0 = sc.render_rays(p, 0, 1)
    assert (r0 == S2).all() and st0["rays_closest"] == n * S2
    e = _pass0_error(m0, e0).ravel()
    key = ray_key(e, 1, r0.ravel(), 0.0)
    values, counts = np.unique(key[key > 0], return_counts=True)
    print(f"{int((key > 0).sum())} candidates in {len(values)} groups of equal keys: {counts[::-1].tolist()}")
    assert counts.max() >= 500
    g = int(np.argmax(counts))
    above = int(counts[g + 1:].sum())
    for K in (above + 1, above + counts[g] // 2, above + counts[g] - 1):
        _, _, samples, rays, st = sc.render_rays(p, n * S2 + K * S2, 2)
        got = _flagged_twice(samples, S2)
        assert np.array_equal(got, select_pixels(e, 0.0, K)) and len(got) == K
        in_group = np.flatnonzero(key == values[g])
        assert np.array_equal(np.intersect1d(got, in_group), in_group[:K - above])  # the lowest pixel indices of the group
        assert st["rays_closest"] == (n + K) * S2 and int(rays.sum()) == st["rays_closest"]


def _replay_rays(means, errs, rays, R, M, target, floor=1e-2, band=1e-6):
    """Host replica of rt_render_adaptive_rays from what every pass gives each pixel ([K][H][W][3] mean and SE, [K][H][W]
    rays of single-pass renders).  The mean in fp32 in pass order and the rays as integers are exact; e and the key of a
    pixel with P >= 2 come from the observable SE in fp64 (test_gpu_budget.py _replay_budget gives the band), with P = 1
    in fp32 exactly.  `ambiguous` counts the decisions an approximate value came within a relative `band` of: the
    target, or the order of two keys next to the cut."""
    K_, H, W, _ = means.shape
    m = means.reshape(K_, -1, 3).astype(np.float32)
    v = errs.reshape(K_, -1, 3).astype(np.float64) ** 2
    nr = rays.reshape(K_, -1).astype(np.int64)
    n = H * W
    sum_m, sum_v, N = m[0].copy(), v[0].copy(), nr[0].copy()
    P = np.ones(n, dtype=np.int64)
    t, fl = float(np.float32(target)), np.float32(floor)
    spent, pixels_in_pass, passes_info, ambiguous, stop = int(N.sum()), [n], [], 0, "passes"
    for p in range(M - 1):
        mean = sum_m / P[:, None].astype(np.float32)
        e = (np.sqrt(sum_v) / P[:, None] / np.maximum(mean, fl)).max(-1)
        exact = P == 1
        w = predicted_cost(N, P)
        key = np.where(e > t, np.maximum(e / np.sqrt((P + 1.0) * w), float(FLT_MIN)), 0.0)
        key[exact] = ray_key(e[exact].astype(np.float32), P[exact], w[exact], target)
        if t > 0:
            ambiguous += int((~exact & (np.abs(e / t - 1.0) < band)).sum())
        cand = np.flatnonzero(key > 0)
        W_c, R_left = int(w[cand].sum()), R - spent
        T = spend_target(R_left, W_c, M - 1 - p)
        order = cand[np.lexsort((cand, -key[cand]))]
        take = int(np.searchsorted(np.cumsum(w[order]), T, side="right"))
        for a in (take - 1, take):  # the pixel left out first, against its neighbours in the order
            if 0 <= a and a + 1 < len(order):
                i, j = order[a], order[a + 1]
                if not (exact[i] and exact[j]) and key[i] - key[j] <= band * key[i]:
                    ambiguous += 1
        sel = np.sort(order[:take])
        actual = int(nr[p + 1][sel].sum())
        passes_info.append(dict(R_left=R_left, W_c=W_c, T=T, cost=int(w[sel].sum()), actual=actual,
                                w_max=int(w[cand].max()) if len(cand) else 0))
        if take == 0:
            stop = "empty"
            break
        sum_m[sel] = sum_m[sel] + m[p + 1][sel]
        sum_v[sel] += v[p + 1][sel]
        N[sel] += nr[p + 1][sel]
        P[sel] += 1
        spent += actual
        pixels_in_pass.append(take)
    return dict(mean=(sum_m / P[:, None].astype(np.float32)).reshape(H, W, 3), P=P.reshape(H, W), N=N.reshape(H, W), spent=spent,
                pixels_in_pass=pixels_in_pass, passes=passes_info, ambiguous=ambiguous, stop=stop)


@pytest.mark.parametrize("budget, max_passes, target", [(0.5, 4, 0.0), (2.5, 4, 0.0), (4.0, 6, 0.0), (3.0, 5, 0.03),
                                                        (1.6, 2, 0.0), (8.0, 3, 0.05)])
def test_passes_replay_on_the_host_within_the_budget(budget, max_passes, target):
    """S^2 = 64: one pixel per task, so a pixel's pass values do not depend on the list it is traced in."""
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    S, W, H = 8, 160, 120
    S2 = S * S
    means, errs, rays = [], [], []
    for pas in range(max_passes):
        mp, ep, _, rp, _ = sc.render_rays(_params(W, H, cam, S, pas), 0, 1)
        means.append(mp)
        errs.append(ep)
        rays.append(rp)
    R = int(budget * int(rays[0].sum()))
    # a target that no approximate e of the replay lies within the band of (chosen on the host, before the device call)
    for t in ([target] if target == 0 else [target * f for f in (1.0, 0.97, 1.03, 0.94, 1.06)]):
        r = _replay_rays(np.stack(means), np.stack(errs), np.stack(rays), R, max_passes, t)
        if r["ambiguous"] == 0:
            target = t
            break
    mean, err, samples, got_rays, st = sc.render_rays(_params(W, H, cam, S), R, max_passes, target)
    print(f"R = {budget} x pass 0 = {R}, M {max_passes}, target {target}: pixels per pass {st['pixels_in_pass']} (host "
          f"{r['pixels_in_pass']}), {st['rays_closest']} rays spent, stop: {r['stop']}; per pass "
          f"{[(q['R_left'], q['T'], q['cost'], q['actual']) for q in r['passes']]}")
    assert r["ambiguous"] == 0  # so that the comparison below means something
    assert st["pixels_in_pass"] == r["pixels_in_pass"] and st["passes"] == len(r["pixels_in_pass"])
    assert np.array_equal(samples // S2, r["P"]) and (samples % S2 == 0).all() and (samples <= max_passes * S2).all()
    assert np.array_equal(mean, r["mean"]) and np.array_equal(got_rays, r["N"])
    assert st["rays_closest"] == int(got_rays.sum()) == r["spent"] and st["overflow"] == 0
    # the stop reason is the rule's: an empty prefix, or M passes
    assert (r["stop"] == "passes") == (st["passes"] == max_passes)
    over = 0
    for q in r["passes"]:
        assert q["cost"] <= max(q["R_left"], 0) and q["cost"] <= q["T"]  # a pass's predicted cost fits what is left
        if q["R_left"] > 0 and q["W_c"] > 0:
            assert q["cost"] >= min(-(-q["W_c"] // 2), q["R_left"]) - q["w_max"]  # at least half the candidates' cost
        over += max(q["actual"] - q["cost"], 0)
    # the rays spent exceed R only by the passes' overrun of their prediction, or by pass 0 alone
    assert st["rays_closest"] <= max(R, int(rays[0].sum())) + over
    if budget < 1:
        assert st["passes"] == 1 and r["stop"] == "empty"


def test_deterministic_and_leaves_the_streams_where_plain_renders_do():
    world, camera = scenes.demo_scene()

    def run():
        tracer = CudaImageTracer(HdrImage(160, 120), camera, samples_per_side=4, pcg=PCG(42, 54))
        renderer = PathTracer(world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3)
        first = CudaImageTracer(HdrImage(160, 120), camera, samples_per_side=4, pcg=PCG(42, 54))
        first.fire_all_rays(PathTracer(world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3))
        mean_rays = 3.0 * first.last_stats["rays_closest"] / (160 * 120)
        res = tracer.fire_all_rays_adaptive(renderer, mean_rays_per_pixel=mean_rays, max_samples_per_pixel=160)
        return tracer, renderer, res, mean_rays

    tracer, renderer, res, mean_rays = run()
    again = run()
    assert np.array_equal(tracer.image.rgb_array(), again[0].image.rgb_array())
    assert np.array_equal(res.error, again[2].error) and np.array_equal(res.samples, again[2].samples)
    assert np.array_equal(res.rays, again[2].rays)
    assert all(res.stats[k] == again[2].stats[k] for k in ("rays_closest", "samples", "passes", "pixels_in_pass", "ray_budget"))
    assert res.passes >= 3 and res.stats["ray_budget"] == int(np.floor(mean_rays * 160 * 120))
    assert res.rays.shape == (120, 160) and int(res.rays.sum()) == res.stats["rays_closest"]
    plain_t = CudaImageTracer(HdrImage(160, 120), camera, samples_per_side=4, pcg=PCG(42, 54))
    plain_r = PathTracer(world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3)
    for _ in range(res.passes):
        plain_t.fire_all_rays(plain_r)
    assert (tracer.pcg.state, renderer.pcg.state) == (plain_t.pcg.state, plain_r.pcg.state)


def test_render_command_writes_the_in_process_image(tmp_path):
    from click.testing import CliRunner

    from pytracer_b200.hdrimage import read_pfm_image
    from pytracer_b200.main import cli

    scene = tmp_path / "demo.txt"
    scene.write_text(DEMO_TXT)
    parsed = parse_scene_text(DEMO_TXT)
    image = HdrImage(96, 72)
    tracer = CudaImageTracer(image, parsed.camera, samples_per_side=4)
    one = CudaImageTracer(HdrImage(96, 72), parsed.camera, samples_per_side=4)
    one.fire_all_rays(PathTracer(parsed.world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3))
    mean_rays = repr(2.5 * one.last_stats["rays_closest"] / (96 * 72))  # two and a half uniform passes
    renderer = PathTracer(parsed.world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3)
    res = tracer.fire_all_rays_adaptive(renderer, mean_rays_per_pixel=float(mean_rays), max_samples_per_pixel=128,
                                        error_estimator="paired")
    with open(tmp_path / "inproc.pfm", "wb") as f:
        image.write_pfm(f)
    out = {k: tmp_path / f"{k}" for k in ("img.pfm", "img.png", "err.pfm")}
    result = CliRunner().invoke(cli, ["render", "--width", "96", "--height", "72", "--samples-per-pixel", "16",
                                      "--mean-rays-per-pixel", mean_rays, "--max-samples-per-pixel", "128",
                                      "--error-estimator", "paired", "--pfm-output", str(out["img.pfm"]),
                                      "--png-output", str(out["img.png"]), "--error-output", str(out["err.pfm"]), str(scene)])
    print(result.output)
    assert result.exit_code == 0, result.output
    assert all(p.exists() and p.stat().st_size > 0 for p in out.values())
    assert f"budget {res.stats['ray_budget']} rays, {res.stats['rays_closest']} spent" in result.output
    assert (tmp_path / "inproc.pfm").read_bytes() == out["img.pfm"].read_bytes()
    assert res.passes >= 2
    with open(out["err.pfm"], "rb") as f:
        err = read_pfm_image(f)
    assert np.allclose(err.rgb_array(), res.error)
