"""rt_render_adaptive / CudaImageTracer.fire_all_rays_adaptive on the device: the error-map kernels store
rt_render's image bit for bit, the reported standard errors are calibrated, pass p equals the (p+1)-th plain
render, and noise-targeted passes give a converged, deterministic image that agrees with the oracle."""
import numpy as np
import pytest

from oracle import oracle
from pytracer_b200 import _abi, _native, scenes
from pytracer_b200.device import DeviceScene
from pytracer_b200.flatten import flatten_world
from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.imagetracer import CudaImageTracer
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG
from pytracer_b200.render import PathTracer
from util import assert_luminance_agreement, assert_mc_agreement, demo_flat

pytestmark = pytest.mark.gpu

PT = dict(algorithm="pathtracing", num_of_rays=10, max_depth=3, rr_limit=3)


def _relative_error(mean, se, floor=1e-2):
    return (se / np.maximum(mean, floor)).max(-1)


@pytest.mark.parametrize("case", ["demo 64 spp", "demo 16 spp", "spheres37 16 spp", "spheres37 16 spp bvh"])
def test_error_map_leaves_the_image_bit_identical(case):
    if case.startswith("demo"):
        fs, cam = demo_flat()
        kw = dict(PT)
    else:
        rs = scenes.random_spheres_scene(37)
        fs, cam = flatten_world(rs.world), rs.camera
        kw = dict(algorithm="pathtracing", num_of_rays=4, max_depth=3, rr_limit=2, accel="bvh" if "bvh" in case else "none")
    S = 8 if "64" in case else 4
    sc = DeviceScene(fs)
    p = make_params(160, 120, cam, samples_per_side=S, aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54), **kw)
    rgb, _, st = sc.render(p)
    mean, err, samples, ast = sc.render_adaptive(p, 0.0, 1)
    assert np.array_equal(mean, rgb), case
    assert (samples == S * S).all() and ast["passes"] == 1 and ast["pixels_in_pass"] == [160 * 120]
    assert (ast["rays_closest"], ast["samples"]) == (st["rays_closest"], st["samples"]) and ast["overflow"] == 0
    assert np.isfinite(err).all() and (err >= 0).all()


@pytest.mark.parametrize("S", [8, 4])
def test_reported_standard_error_is_calibrated(S):
    """K = 16 independent single-pass renders of demo.txt: the mean reported SE^2 against the variance of the
    run means, and the spread of the runs in units of their own reported SE."""
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    runs, ses = [], []
    for k in range(16):
        p = make_params(160, 120, cam, samples_per_side=S, aa_pcg=PCG(1000 + k, 7), pt_pcg=PCG(2000 + k, 9), **PT)
        mean, err, _, _ = sc.render_adaptive(p, 0.0, 1)
        runs.append(mean.astype(np.float64))
        ses.append(err.astype(np.float64))
    runs, ses = np.stack(runs), np.stack(ses)
    var_emp = runs.var(0, ddof=1)
    agree = (runs == runs[0]).all(0)  # values whose samples all agree (misses, the sky seen directly)
    assert (ses[:, agree] <= 1e-6 * np.abs(runs[:, agree])).all()
    n_const = int(agree.all(-1).sum())
    print(f"S = {S}: {n_const} pixels without variance (anchor 9 388)")
    assert abs(n_const - 9388) <= 0.01 * 9388
    noisy = var_emp > 1e-12 * np.maximum(runs.mean(0) ** 2, 1e-6)
    ratio = np.median((ses ** 2).mean(0)[noisy] / var_emp[noisy])
    z = (runs - runs.mean(0)) / np.where(ses > 0, ses, np.inf)
    frac = float((np.abs(z[:, noisy]) <= 3.0).mean())
    print(f"S = {S}: {int(noisy.sum())} noisy values, median SE^2 / var = {ratio:.3f}, |z| <= 3 for {frac:.4f}")
    # The batch estimator treats the S^2 stratified samples as independent; stratification removes the part of the
    # variance that comes from where in the pixel a sample lands, so the reported SE^2 is an upper bound.  On
    # demo.txt at 64 spp it is 1.54x the variance of the run means (B200, DESIGN.md §5.5): conservative, and the
    # convergence test errs towards more samples, never fewer.
    # A pass's SE comes from B = 32 (64 spp) or 16 (16 spp) batch sums, so z follows Student's t with B - 1 degrees
    # of freedom at best (P(|t_15| <= 3) = 0.991), and the skewed per-sample distribution of a path tracer widens
    # the tails further (measured: 0.995 at 64 spp, 0.981 at 16 spp)
    assert 0.8 <= ratio <= 2.0
    assert frac >= (0.99 if S * S >= 64 else 0.975)


@pytest.mark.parametrize("S", [8, 4])
def test_passes_equal_successive_plain_renders(S):
    world, camera = scenes.demo_scene()
    plain = []
    tracer = CudaImageTracer(HdrImage(160, 120), camera, samples_per_side=S, pcg=PCG(42, 54))
    renderer = PathTracer(world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3)
    states = [(tracer.pcg.state, renderer.pcg.state)]
    for _ in range(3):
        tracer.fire_all_rays(renderer)
        plain.append(tracer.image.rgb_array().copy())
        states.append((tracer.pcg.state, renderer.pcg.state))
    tracer = CudaImageTracer(HdrImage(160, 120), camera, samples_per_side=S, pcg=PCG(42, 54))
    renderer = PathTracer(world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3)
    res = tracer.fire_all_rays_adaptive(renderer, target_error=0.03, max_samples_per_pixel=3 * S * S)
    n = res.stats["pixels_in_pass"]
    print(f"S = {S}: pixels per pass {n}")
    assert res.passes == 3 and n[0] > n[1] > n[2] > 0
    P = res.samples // (S * S)
    got = tracer.image.rgb_array()
    expect = {1: plain[0], 2: (plain[0] + plain[1]) / np.float32(2), 3: ((plain[0] + plain[1]) + plain[2]) / np.float32(3)}
    for p in (1, 2, 3):
        sel = P == p
        assert sel.any()
        if S * S >= 32:  # one pixel per task: the same sums in the same order
            assert np.array_equal(got[sel], expect[p][sel]), p
        else:  # pixels of one task differ from pass to pass: equal to fp32 rounding
            assert np.allclose(got[sel], expect[p][sel], rtol=1e-5, atol=1e-7), p
    assert (tracer.pcg.state, renderer.pcg.state) == states[res.passes]


def _oracle_runs(fs, cam, runs):
    import os

    threads = max(1, min(32, os.cpu_count() or 1))
    return np.stack([oracle.render_threaded(fs, make_params(160, 120, cam, samples_per_side=4, aa_pcg=PCG(1000 + k, 7),
                                                            pt_pcg=PCG(2000 + k, 9), **PT), threads)["rgb"].copy()
                     for k in range(runs)])


def test_adaptive_image_meets_its_target_and_agrees_with_the_reference_estimator():
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    p = make_params(160, 120, cam, samples_per_side=4, aa_pcg=PCG(11, 3), pt_pcg=PCG(77, 5), **PT)
    mean, err, samples, st = sc.render_adaptive(p, 0.02, 64)
    pass0, _, _ = sc.render(p)
    e = _relative_error(mean.astype(np.float64), err.astype(np.float64))
    print(f"adaptive demo.txt: passes {st['passes']}, pixels per pass {st['pixels_in_pass']}, "
          f"{st['samples']} samples ({st['samples'] / samples.size:.1f} per pixel), {st['kernel_ms']:.2f} ms")
    assert ((e <= 0.02) | (samples == 1024)).all()
    flat = (err == 0).all(-1)
    assert flat.sum() > 0 and (samples[flat] == 16).all() and np.array_equal(mean[flat], pass0[flat])
    # counters add up
    assert st["samples"] == int(samples.sum()) and st["overflow"] == 0
    assert len(st["pixels_in_pass"]) == min(st["passes"], 16) and st["pixels_in_pass"][0] == samples.size
    if st["passes"] <= 16:
        assert st["samples"] == sum(st["pixels_in_pass"]) * 16
    assert (np.bincount((samples // 16).ravel())[1:] >= 0).all() and int((samples >= 16 * 2).sum()) == st["pixels_in_pass"][1]
    assert st["rays_closest"] >= st["samples"]
    # deterministic
    again = sc.render_adaptive(p, 0.02, 64)
    assert np.array_equal(again[0], mean) and np.array_equal(again[1], err) and np.array_equal(again[2], samples)
    # the 24 x 16-spp oracle runs of test_streams_agree_statistically_with_the_reference_estimator
    ref = _oracle_runs(fs, cam, 24)
    gpu = mean.astype(np.float64)
    assert_luminance_agreement(gpu, ref, what="adaptive demo.txt 160x120")
    assert_mc_agreement(gpu, ref, samples_ratio=(24 * 16) / samples[..., None].astype(np.float64), n_ref=24 * 16,
                        what="adaptive demo.txt 160x120")


def test_calls_outside_the_scope_are_refused():
    fs, cam = demo_flat()
    sc = DeviceScene(fs)
    base = dict(samples_per_side=4, **PT)
    bad = [dict(base, algorithm="flat"), dict(base, samples_per_side=1), dict(base, variant="mega"), dict(base, precision="f64"),
           dict(base, part_mode=_abi.RT_PART_SPP, part_count=2), dict(base, out_f64=True), dict(base, rng_mode=_abi.RT_RNG_REPLAY)]
    for kw in bad:
        with pytest.raises(_native.NativeError) as e:
            sc.render_adaptive(make_params(32, 24, cam, **kw), 0.05, 4)
        assert e.value.code == _abi.RT_ERR_INVALID, kw
    with pytest.raises(_native.NativeError) as e:
        sc.render_adaptive(make_params(32, 24, cam, **base), 0.05, 0)
    assert e.value.code == _abi.RT_ERR_INVALID


def test_render_command_writes_image_and_error_map(tmp_path):
    from click.testing import CliRunner

    from pytracer_b200.hdrimage import read_pfm_image
    from pytracer_b200.main import cli
    from test_adaptive_cpu import DEMO_TXT

    scene = tmp_path / "demo.txt"
    scene.write_text(DEMO_TXT)
    out = {k: tmp_path / f"{k}" for k in ("img.pfm", "img.png", "err.pfm")}
    result = CliRunner().invoke(cli, ["render", "--width", "96", "--height", "72", "--samples-per-pixel", "16",
                                      "--target-error", "0.05", "--max-samples-per-pixel", "128",
                                      "--pfm-output", str(out["img.pfm"]), "--png-output", str(out["img.png"]),
                                      "--error-output", str(out["err.pfm"]), str(scene)])
    print(result.output)
    assert result.exit_code == 0, result.output
    assert all(p.exists() and p.stat().st_size > 0 for p in out.values())
    assert "pass(es)" in result.output
    # the same call in-process, from the same defaults as the command (--init-state 45, --init-seq 54)
    from pytracer_b200.scene_text import parse_scene_text

    parsed = parse_scene_text(DEMO_TXT)
    image = HdrImage(96, 72)
    tracer = CudaImageTracer(image, parsed.camera, samples_per_side=4)
    res = tracer.fire_all_rays_adaptive(PathTracer(parsed.world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3),
                                        target_error=0.05, max_samples_per_pixel=128)
    with open(tmp_path / "inproc.pfm", "wb") as f:
        image.write_pfm(f)
    assert (tmp_path / "inproc.pfm").read_bytes() == out["img.pfm"].read_bytes()
    with open(out["err.pfm"], "rb") as f:
        err = read_pfm_image(f)
    assert np.allclose(err.rgb_array(), res.error)
