"""Sample-budget rendering without a device: the argument checks of fire_all_rays_adaptive(mean_samples_per_pixel=...)
(ValueError before any device call), the `render --mean-samples-per-pixel` option refusing what it cannot run, and the
host replica of the rule that sizes and fills every pass after the first (rt_render_adaptive_budget, include/rt_api.h),
which tests/test_gpu_budget.py compares the device with."""
import numpy as np
import pytest
from click.testing import CliRunner

from pytracer_b200 import scenes
from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.imagetracer import CudaImageTracer
from pytracer_b200.main import adaptive_cli_problem, cli
from pytracer_b200.pcg import PCG
from pytracer_b200.render import FlatRenderer, PathTracer
from test_adaptive_cpu import DEMO_TXT


def pass_size(C, Q, r):
    """K = min(C, Q, max(ceil(C / 2), ceil(Q / r))): C candidates, Q pixel passes the budget still pays for, r passes left."""
    return min(C, Q, max(-(-C // 2), -(-Q // r)))


def select_pixels(e, target, K):
    """The first K pixels with e > target in the order (e descending, pixel index ascending), in ascending order.
    `e`: float32 per pixel (any shape, flattened in C order)."""
    e = np.asarray(e, dtype=np.float32).ravel()
    cand = np.flatnonzero(e > np.float32(target))
    order = cand[np.lexsort((cand, -e[cand].astype(np.float64)))]
    return np.sort(order[:K])


def test_pass_size_rule_by_hand():
    assert pass_size(1000, 3000, 4) == 750  # ceil(Q / r): the budget spread over the passes left
    assert pass_size(1000, 1000, 4) == 500  # at least half of the candidates
    assert pass_size(100, 1000, 4) == 100  # every candidate
    assert pass_size(101, 1000, 9) == 101 and pass_size(101, 40, 9) == 40
    # the last allowed pass (r = 1) spends the rest of the budget, or traces every candidate
    assert pass_size(100, 37, 1) == 37 and pass_size(10, 37, 1) == 10
    # no candidates, or no budget: the call stops
    assert pass_size(0, 500, 3) == 0 and pass_size(50, 0, 3) == 0 and pass_size(0, 0, 1) == 0
    # Q below ceil(C / 2): the budget bounds the pass
    assert pass_size(100, 20, 5) == 20 and pass_size(7, 3, 2) == 3
    # odd counts round up
    assert pass_size(7, 100, 50) == 4 and pass_size(9, 10, 3) == 5


def test_selection_orders_by_error_then_index():
    e = np.array([0.5, 0.1, 0.5, 0.0, 0.3, 0.5, 0.2], dtype=np.float32)
    assert select_pixels(e, 0.0, 2).tolist() == [0, 2]  # the cut inside the tie group {0, 2, 5}: lowest index first
    assert select_pixels(e, 0.0, 4).tolist() == [0, 2, 4, 5]
    assert select_pixels(e, 0.0, 99).tolist() == [0, 1, 2, 4, 5, 6]  # pixel 3 has no error
    assert select_pixels(e, 0.25, 99).tolist() == [0, 2, 4, 5]  # only candidates
    assert select_pixels(e, 0.5, 3).tolist() == [] and select_pixels(e, 0.0, 0).tolist() == []


def _tracer(samples_per_side=4):
    world, camera = scenes.demo_scene()
    return CudaImageTracer(HdrImage(8, 6), camera, samples_per_side=samples_per_side), world


@pytest.mark.parametrize("case, kwargs, match", [
    ("mean below one pass", {"mean_samples_per_pixel": 8, "max_samples_per_pixel": 64}, "at least the samples of the first pass"),
    ("mean not an integer", {"mean_samples_per_pixel": 20.5, "max_samples_per_pixel": 64}, "integer"),
    ("max missing", {"mean_samples_per_pixel": 32}, "max_samples_per_pixel"),
    ("max below the mean", {"mean_samples_per_pixel": 48, "max_samples_per_pixel": 32}, "max_samples_per_pixel >= the mean"),
    ("max not a multiple of S^2", {"mean_samples_per_pixel": 32, "max_samples_per_pixel": 40}, "multiple"),
    ("flat renderer", {"mean_samples_per_pixel": 32, "max_samples_per_pixel": 64}, "path-tracing"),
    ("two GPUs", {"mean_samples_per_pixel": 32, "max_samples_per_pixel": 64, "gpus": 2}, "one device"),
    ("mega variant", {"mean_samples_per_pixel": 32, "max_samples_per_pixel": 64, "variant": "mega"}, "warp"),
    ("fp64", {"mean_samples_per_pixel": 32, "max_samples_per_pixel": 64, "precision": "f64"}, "warp"),
    ("negative target", {"mean_samples_per_pixel": 32, "max_samples_per_pixel": 64, "target_error": -0.1}, "target_error"),
    ("NaN target", {"mean_samples_per_pixel": 32, "max_samples_per_pixel": 64, "target_error": float("nan")}, "target_error"),
    ("odd S with the paired estimator", {"mean_samples_per_pixel": 36, "max_samples_per_pixel": 72, "samples_per_side": 3,
                                         "error_estimator": "paired"}, "even"),
])
def test_budget_arguments_are_checked_before_any_device_call(case, kwargs, match):
    kwargs = dict(kwargs)
    tracer, world = _tracer(kwargs.pop("samples_per_side", 4))
    renderer_kw = {k: kwargs.pop(k) for k in ("variant", "precision", "gpus") if k in kwargs}
    renderer = FlatRenderer(world) if case == "flat renderer" else PathTracer(world, pcg=PCG(45, 54), **renderer_kw)
    pcg_before = (tracer.pcg.state, renderer.pcg.state)
    with pytest.raises(ValueError, match=match):
        tracer.fire_all_rays_adaptive(renderer, **kwargs)
    assert renderer._scene is None  # nothing reached the device
    assert (tracer.pcg.state, renderer.pcg.state) == pcg_before


@pytest.mark.parametrize("args, message", [
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "32"], "needs --max-samples-per-pixel"),
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "32", "--target-error", "0.05"], "needs --max-samples-per-pixel"),
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "8", "--max-samples-per-pixel", "64"], "must be at least --samples-per-pixel"),
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "96", "--max-samples-per-pixel", "64"], "must be at least --mean-samples"),
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "32", "--max-samples-per-pixel", "40"], "multiple"),
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "32", "--max-samples-per-pixel", "64", "--target-error", "-1"],
     "target-error"),
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "32", "--max-samples-per-pixel", "64", "--target-error", "nan"],
     "target-error"),
    (["--algorithm", "flat", "--mean-samples-per-pixel", "32", "--max-samples-per-pixel", "64"], "pathtracing"),
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "32", "--max-samples-per-pixel", "64", "--gpus", "2"], "one GPU"),
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "32", "--max-samples-per-pixel", "64", "--variant", "mega"], "warp"),
    (["--samples-per-pixel", "16", "--mean-samples-per-pixel", "32", "--max-samples-per-pixel", "64", "--precision", "f64"], "warp"),
    (["--samples-per-pixel", "9", "--mean-samples-per-pixel", "18", "--max-samples-per-pixel", "36", "--error-estimator", "paired"],
     "even"),
])
def test_render_command_refuses_budget_combinations_it_cannot_run(tmp_path, args, message):
    scene = tmp_path / "demo.txt"
    scene.write_text(DEMO_TXT)
    result = CliRunner().invoke(cli, ["render", "--width", "8", "--height", "6", "--pfm-output", str(tmp_path / "o.pfm"),
                                      "--png-output", str(tmp_path / "o.png"), *args, str(scene)])
    assert result.exit_code != 0, result.output
    assert "Error," in result.output and message in result.output, result.output
    assert not (tmp_path / "o.pfm").exists()


def test_budget_options_that_can_run_pass_the_checks():
    common = ("pathtracing", 16, 1, "auto", "auto")
    for target in (None, 0.0, 0.05):
        assert adaptive_cli_problem(*common, target, 64, 1e-2, "batch", mean_samples_per_pixel=32) is None
    assert adaptive_cli_problem(*common, None, 32, 1e-2, "paired", mean_samples_per_pixel=32) is None
    # without the new option the pairing rule of the threshold mode is unchanged
    assert adaptive_cli_problem(*common, None, 64, 1e-2) == "--target-error and --max-samples-per-pixel go together"
