"""The paired-strata error estimator without a device: its fp64 host reference (tests/paired_ref.py) on synthetic
stratified pixels, the C-ABI field that selects it, and the argument checks of fire_all_rays_adaptive and of the
`render` command (refused before any device call)."""
import ctypes
import os
import subprocess
import tempfile
import textwrap

import numpy as np
import pytest
from click.testing import CliRunner

from paired_ref import paired_se2
from pytracer_b200 import _abi, scenes
from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.imagetracer import CudaImageTracer
from pytracer_b200.main import cli
from pytracer_b200.pcg import PCG
from pytracer_b200.render import PathTracer
from test_adaptive_cpu import DEMO_TXT
from util import batch_se2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _stratified_pixels(f, S, n, rng):
    """n independent passes over one pixel: sample ls = row * S + column jittered inside its stratum, value f(u, v)."""
    ir, ic = np.divmod(np.arange(S * S), S)
    u = (ic + rng.random((n, S * S))) / S
    v = (ir + rng.random((n, S * S))) / S
    return f(u, v, rng)


def test_paired_se2_matches_a_direct_sum_and_is_unbiased_for_independent_samples():
    rng = np.random.default_rng(5)
    x = rng.normal(size=(3, 36))
    T = np.array([x[:, b::32].sum(-1) for b in range(32)]).T   # bpp 32: batch sums, uneven sizes (2 or 1)
    want = sum((T[:, 2 * j] - T[:, 2 * j + 1]) ** 2 for j in range(16)) / 36 ** 2
    se2, bound = paired_se2(x, 32, bound=True)
    assert np.allclose(se2, want, rtol=1e-12, atol=0) and (bound > 0).all()
    assert np.allclose(paired_se2(x[:, :4], 4), ((x[:, 0] - x[:, 1]) ** 2 + (x[:, 2] - x[:, 3]) ** 2) / 16, rtol=1e-12)
    for L, bpp in ((4, 4), (16, 16), (36, 32), (64, 32), (256, 32)):
        x = rng.normal(0.0, 1.5, size=(min(200_000, 4_000_000 // L), L))
        ratio = paired_se2(x, bpp).mean() / (1.5 ** 2 / L)
        print(f"L = {L}, bpp = {bpp}: mean SE^2 / (sigma^2 / L) = {ratio:.4f}")
        assert abs(ratio - 1.0) <= 0.01, (L, bpp, ratio)
    with pytest.raises(AssertionError):
        paired_se2(np.zeros((2, 9)), 32)


def _true_var(f, S, rng, n=200_000):
    return _stratified_pixels(f, S, n, rng).mean(-1).var()


@pytest.mark.parametrize("S, bpp", [(2, 4), (4, 16), (6, 32), (8, 32)])
def test_paired_is_conservative_and_below_the_batch_estimator_on_a_smooth_gradient(S, bpp):
    """Radiance a + b u + c v plus noise: the pair difference of two neighbouring strata carries b / S of slope,
    so the estimate stays above the variance of the stratified mean, and below the batch estimator, which counts
    the whole spread of the gradient over the pixel as noise (at S = 2 only just: there the horizontal slope
    between two neighbours is half the pixel's)."""
    rng = np.random.default_rng(S)
    f = lambda u, v, r: 0.5 + 0.8 * u + 0.6 * v + r.normal(0.0, 0.05, u.shape)
    x = _stratified_pixels(f, S, 100_000, rng)
    true = _true_var(f, S, rng)
    paired, batch = paired_se2(x, bpp).mean(), batch_se2(x, bpp).mean()
    print(f"S = {S}: true {true:.3e}, paired {paired:.3e} ({paired / true:.2f}x), batch {batch:.3e} ({batch / true:.2f}x)")
    assert paired >= 0.99 * true
    assert paired < 0.98 * batch


@pytest.mark.parametrize("edge", ["vertical at u = 0.37", "vertical on a stratum border", "horizontal at v = 0.61",
                                  "diagonal"])
def test_paired_stays_conservative_on_a_step_edge_inside_the_pixel(edge):
    rng = np.random.default_rng(11)
    step = {"vertical at u = 0.37": lambda u, v: u > 0.37, "vertical on a stratum border": lambda u, v: u > 0.5,
            "horizontal at v = 0.61": lambda u, v: v > 0.61, "diagonal": lambda u, v: u + 0.7 * v > 0.8}[edge]
    for S, bpp in ((2, 4), (4, 16), (8, 32)):
        f = lambda u, v, r: np.where(step(u, v), 1.0, 0.1) + r.normal(0.0, 0.01, u.shape)
        x = _stratified_pixels(f, S, 100_000, rng)
        true = _true_var(f, S, rng)
        paired = paired_se2(x, bpp)
        print(f"{edge}, S = {S}: mean paired SE^2 / Var(mean) = {paired.mean() / true:.3f}")
        assert paired.mean() >= 0.98 * true, (S, paired.mean() / true)


def test_estimator_field_keeps_the_struct_layout():
    src = textwrap.dedent("""
        #include <stddef.h>
        #include <stdio.h>
        #include "rt_api.h"
        int main(void) {
          printf("%zu %zu %d %d\\n", sizeof(rt_adaptive_params), offsetof(rt_adaptive_params, estimator),
                 RT_ERR_EST_BATCH, RT_ERR_EST_PAIRED);
          return 0;
        }""")
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "s")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    P = _abi.rt_adaptive_params
    assert got == [ctypes.sizeof(P), P.estimator.offset, _abi.RT_ERR_EST_BATCH, _abi.RT_ERR_EST_PAIRED] == [24, 20, 0, 1]
    assert _abi.ERROR_ESTIMATORS == {"batch": _abi.RT_ERR_EST_BATCH, "paired": _abi.RT_ERR_EST_PAIRED}


@pytest.mark.parametrize("S, estimator, match", [(3, "paired", "even samples_per_side"),
                                                 (5, "paired", "even samples_per_side"),
                                                 (4, "stratified", "error_estimator must be one of"),
                                                 (4, "PAIRED", "error_estimator must be one of")])
def test_fire_all_rays_adaptive_refuses_estimators_it_cannot_run_before_any_device_call(S, estimator, match):
    world, camera = scenes.demo_scene()
    tracer = CudaImageTracer(HdrImage(8, 6), camera, samples_per_side=S)
    renderer = PathTracer(world, pcg=PCG(45, 54))
    pcg_before = (tracer.pcg.state, renderer.pcg.state)
    with pytest.raises(ValueError, match=match):
        tracer.fire_all_rays_adaptive(renderer, error_estimator=estimator)
    assert renderer._scene is None  # nothing reached the device
    assert (tracer.pcg.state, renderer.pcg.state) == pcg_before


@pytest.mark.parametrize("args, message", [
    (["--samples-per-pixel", "9", "--error-output", "e.pfm", "--error-estimator", "paired"], "even number of samples"),
    (["--samples-per-pixel", "25", "--target-error", "0.05", "--max-samples-per-pixel", "100", "--error-estimator", "paired"],
     "even number of samples"),
    (["--samples-per-pixel", "9", "--error-estimator", "paired"], "applies to --error-output"),
    (["--samples-per-pixel", "16", "--error-estimator", "paired"], "applies to --error-output"),
    (["--samples-per-pixel", "16", "--error-output", "e.pfm", "--error-estimator", "pairs"], "Invalid value"),
])
def test_render_command_refuses_the_paired_estimator_where_it_cannot_run(tmp_path, args, message):
    scene = tmp_path / "demo.txt"
    scene.write_text(DEMO_TXT)
    result = CliRunner().invoke(cli, ["render", "--width", "8", "--height", "6", "--pfm-output", str(tmp_path / "o.pfm"),
                                      "--png-output", str(tmp_path / "o.png"), *args, str(scene)])
    assert result.exit_code != 0, result.output
    assert message in result.output, result.output
    assert not (tmp_path / "o.pfm").exists()
