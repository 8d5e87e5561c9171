"""Ray-budget rendering without a device: the host replica of the rule that sizes and fills every pass after the first
(rt_render_adaptive_rays, include/rt_api.h), which tests/test_gpu_ray_budget.py compares the device with, checked on
hand-made cases; the argument checks of fire_all_rays_adaptive(mean_rays_per_pixel=...) (ValueError before any device
call); and the `render --mean-rays-per-pixel` option refusing what it cannot run."""
import numpy as np
import pytest
from click.testing import CliRunner

from pytracer_b200 import scenes
from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.imagetracer import AdaptiveResult, CudaImageTracer
from pytracer_b200.main import adaptive_cli_problem, cli
from pytracer_b200.pcg import PCG
from pytracer_b200.render import FlatRenderer, PathTracer
from test_adaptive_cpu import DEMO_TXT
from test_budget_cpu import pass_size, select_pixels

FLT_MIN = np.float32(np.finfo(np.float32).tiny)  # 2^-126


def predicted_cost(n, P):
    """w = ceil(n / P): the rays one more pass of a pixel is predicted to cost (n rays over P passes, integers)."""
    n, P = np.asarray(n, dtype=np.int64), np.asarray(P, dtype=np.int64)
    return -(-n // P)


def ray_key(e, P, w, target):
    """The device's fp32 key: e > target ? max(e / sqrt((P + 1) w), FLT_MIN) : 0, every operation correctly rounded in
    fp32 as __fmul_rn, __fsqrt_rn and __fdiv_rn round."""
    e = np.asarray(e, dtype=np.float32)
    P1 = (np.asarray(P, dtype=np.int64) + 1).astype(np.float32)
    wf = np.asarray(w, dtype=np.int64).astype(np.float32)
    with np.errstate(under="ignore"):
        k = np.maximum(e / np.sqrt(P1 * wf), FLT_MIN)
    return np.where(e > np.float32(target), k, np.float32(0)).astype(np.float32)


def spend_target(R_left, W_c, r):
    """T = min(R_left, max(ceil(W_c / 2), ceil(R_left / r))); R_left <= 0: 0."""
    if R_left <= 0:
        return 0
    return min(R_left, max(-(-W_c // 2), -(-R_left // r)))


def select_prefix(key, w, T):
    """The longest prefix of the order (key descending, pixel index ascending) over the pixels with key > 0 whose sum
    of w is <= T, in ascending pixel order.  `key`: float32 (bits order like the values: all are >= 0)."""
    key = np.asarray(key, dtype=np.float32).ravel()
    w = np.asarray(w, dtype=np.int64).ravel()
    cand = np.flatnonzero(key > 0)
    order = cand[np.lexsort((cand, -key[cand].astype(np.float64)))]
    take = int(np.searchsorted(np.cumsum(w[order]), T, side="right"))  # the first prefix sum above T ends the prefix
    return np.sort(order[:take])


def test_predicted_cost_and_key_by_hand():
    assert predicted_cost([16, 17, 100, 99], [1, 1, 3, 3]).tolist() == [16, 17, 34, 33]
    # e / sqrt((P + 1) w): 0.5 / sqrt(2 * 2) = 0.25 exactly; 0.5 / sqrt(3 * 12) = 0.5 / 6
    assert ray_key([0.5, 0.5], [1, 2], [2, 12], 0.0).tolist() == [0.25, np.float32(np.float32(0.5) / np.float32(6))]
    # a non-candidate's key is 0; a candidate's never falls below FLT_MIN, whatever it costs
    assert ray_key([0.05, 0.0], [1, 1], [16, 16], 0.05).tolist() == [0.0, 0.0]
    tiny = ray_key([np.float32(2.0 ** -140)], [7], [2 ** 30], 0.0)
    assert tiny[0] == FLT_MIN and FLT_MIN == np.float32(2.0 ** -126)
    # the key ranks by e^2 / ((P + 1) w): a pixel that costs four times as much needs twice the error to rank level
    k = ray_key([0.2, 0.4, 0.41], [1, 1, 1], [100, 400, 400], 0.0)
    assert k[0] == k[1] < k[2]


def test_spend_target_by_hand():
    assert spend_target(1000, 600, 4) == 300  # at least half the candidates' predicted cost
    assert spend_target(4000, 600, 4) == 1000  # the budget spread over the passes left
    assert spend_target(100, 600, 4) == 100  # never more than is left
    assert spend_target(0, 600, 4) == 0 and spend_target(-50, 600, 4) == 0  # nothing left: an empty pass
    assert spend_target(777, 10 ** 6, 1) == 777 and spend_target(777, 10, 1) == 777  # r = 1: what is left
    assert spend_target(1000, 7, 9) == 112  # ceil(1000 / 9)


def test_prefix_cut_inside_a_weighted_tie_group():
    key = np.array([0.5, 0.5, 0.5, 0.3, 0.5], dtype=np.float32)
    w = np.array([10, 20, 30, 5, 40])
    # order 0, 1, 2, 4 (ties by index), then 3; prefix sums 10, 30, 60, 100, 105
    assert select_prefix(key, w, 35).tolist() == [0, 1]  # 3 alone would fit, but the prefix ends at pixel 2
    assert select_prefix(key, w, 59).tolist() == [0, 1] and select_prefix(key, w, 60).tolist() == [0, 1, 2]
    assert select_prefix(key, w, 9).tolist() == []  # the first pixel alone costs more: an empty pass
    assert select_prefix(key, w, 104).tolist() == [0, 1, 2, 4]


def test_whole_candidate_set_fits_and_non_candidates_never_count():
    key = np.array([0.0, 0.2, 0.0, 0.1], dtype=np.float32)
    w = np.array([1000, 7, 1000, 9])
    W_c = int(w[key > 0].sum())
    for R_left, r in ((48, 3), (16, 1), (10 ** 9, 2)):
        T = spend_target(R_left, W_c, r)
        assert T >= W_c and select_prefix(key, w, T).tolist() == [1, 3]
    assert select_prefix(key, w, spend_target(-1, W_c, 2)).tolist() == []


def test_unit_weights_reproduce_the_sample_budget_selection():
    """Weight 1 and the target in pixel passes: the same lists as the sample-budget rule (test_budget_cpu)."""
    rng = np.random.default_rng(3)
    for trial in range(200):
        n = int(rng.integers(1, 60))
        e = rng.choice(np.array([0.0, 0.125, 0.25, 0.5, 1.0], dtype=np.float32), n)  # many exact ties
        target = float(rng.choice([0.0, 0.2]))
        Q, r = int(rng.integers(0, 80)), int(rng.integers(1, 6))
        C = int((e > np.float32(target)).sum())
        key = np.where(e > np.float32(target), e, np.float32(0))
        got = select_prefix(key, np.ones(n, dtype=np.int64), spend_target(Q, C, r))
        assert np.array_equal(got, select_pixels(e, target, pass_size(C, Q, r))), trial


def test_the_guarantees_of_a_pass():
    """The predicted cost of a selected pass is <= T <= R_left, and while R_left lasts it is at least
    min(ceil(W_c / 2), R_left) less one pixel's weight."""
    rng = np.random.default_rng(7)
    for trial in range(300):
        n = int(rng.integers(1, 80))
        key = np.where(rng.random(n) < 0.7, rng.random(n).astype(np.float32), np.float32(0))
        w = rng.integers(16, 400, n)
        W_c = int(w[key > 0].sum())
        R_left, r = int(rng.integers(-500, 20000)), int(rng.integers(1, 8))
        T = spend_target(R_left, W_c, r)
        sel = select_prefix(key, w, T)
        cost = int(w[sel].sum())
        assert cost <= max(R_left, 0) and cost <= T
        if R_left > 0 and (key > 0).any():
            assert cost >= min(-(-W_c // 2), R_left) - int(w.max()), trial


def test_adaptive_result_gains_a_trailing_rays_field():
    res = AdaptiveResult(error=np.zeros((1, 1, 3)), samples=np.zeros((1, 1)), passes=1)
    assert res.rays is None and list(AdaptiveResult.__dataclass_fields__)[-1] == "rays"


def _tracer(samples_per_side=4):
    world, camera = scenes.demo_scene()
    return CudaImageTracer(HdrImage(8, 6), camera, samples_per_side=samples_per_side), world


@pytest.mark.parametrize("case, kwargs, match", [
    ("with a sample budget", {"mean_rays_per_pixel": 500.0, "mean_samples_per_pixel": 32, "max_samples_per_pixel": 64},
     "exclude each other"),
    ("max missing", {"mean_rays_per_pixel": 500.0}, "needs max_samples_per_pixel"),
    ("negative mean", {"mean_rays_per_pixel": -1.0, "max_samples_per_pixel": 64}, "finite and >= 0"),
    ("NaN mean", {"mean_rays_per_pixel": float("nan"), "max_samples_per_pixel": 64}, "finite and >= 0"),
    ("infinite mean", {"mean_rays_per_pixel": float("inf"), "max_samples_per_pixel": 64}, "finite and >= 0"),
    ("budget beyond int64", {"mean_rays_per_pixel": 1e30, "max_samples_per_pixel": 64}, "too large"),
    ("max not a multiple of S^2", {"mean_rays_per_pixel": 500.0, "max_samples_per_pixel": 40}, "multiple"),
    ("flat renderer", {"mean_rays_per_pixel": 500.0, "max_samples_per_pixel": 64}, "path-tracing"),
    ("two GPUs", {"mean_rays_per_pixel": 500.0, "max_samples_per_pixel": 64, "gpus": 2}, "one device"),
    ("mega variant", {"mean_rays_per_pixel": 500.0, "max_samples_per_pixel": 64, "variant": "mega"}, "warp"),
    ("negative target", {"mean_rays_per_pixel": 500.0, "max_samples_per_pixel": 64, "target_error": -0.1}, "target_error"),
    ("odd S with the paired estimator", {"mean_rays_per_pixel": 500.0, "max_samples_per_pixel": 72, "samples_per_side": 3,
                                         "error_estimator": "paired"}, "even"),
])
def test_ray_budget_arguments_are_checked_before_any_device_call(case, kwargs, match):
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
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "500"], "needs --max-samples-per-pixel"),
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "500", "--target-error", "0.05"], "needs --max-samples-per-pixel"),
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "500", "--mean-samples-per-pixel", "32", "--max-samples-per-pixel", "64"],
     "exclude each other"),
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "-3", "--max-samples-per-pixel", "64"], "mean-rays-per-pixel must be"),
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "nan", "--max-samples-per-pixel", "64"], "mean-rays-per-pixel must be"),
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "inf", "--max-samples-per-pixel", "64"], "mean-rays-per-pixel must be"),
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "500", "--max-samples-per-pixel", "40"], "multiple"),
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "500", "--max-samples-per-pixel", "64", "--target-error", "-1"],
     "target-error"),
    (["--algorithm", "flat", "--mean-rays-per-pixel", "500", "--max-samples-per-pixel", "64"], "pathtracing"),
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "500", "--max-samples-per-pixel", "64", "--gpus", "2"], "one GPU"),
    (["--samples-per-pixel", "16", "--mean-rays-per-pixel", "500", "--max-samples-per-pixel", "64", "--precision", "f64"], "warp"),
    (["--samples-per-pixel", "9", "--mean-rays-per-pixel", "500", "--max-samples-per-pixel", "36", "--error-estimator", "paired"],
     "even"),
])
def test_render_command_refuses_ray_budget_combinations_it_cannot_run(tmp_path, args, message):
    scene = tmp_path / "demo.txt"
    scene.write_text(DEMO_TXT)
    result = CliRunner().invoke(cli, ["render", "--width", "8", "--height", "6", "--pfm-output", str(tmp_path / "o.pfm"),
                                      "--png-output", str(tmp_path / "o.png"), *args, str(scene)])
    assert result.exit_code != 0, result.output
    assert "Error," in result.output and message in result.output, result.output
    assert not (tmp_path / "o.pfm").exists()


def test_ray_budget_options_that_can_run_pass_the_checks():
    common = ("pathtracing", 16, 1, "auto", "auto")
    for target in (None, 0.0, 0.05):
        for mean in (0.0, 123.5, 4000.0):
            assert adaptive_cli_problem(*common, target, 64, 1e-2, "batch", mean_rays_per_pixel=mean) is None
    assert adaptive_cli_problem(*common, None, 32, 1e-2, "paired", mean_rays_per_pixel=500.0) is None
    # the other modes' rules are unchanged
    assert adaptive_cli_problem(*common, None, 64, 1e-2) == "--target-error and --max-samples-per-pixel go together"
    assert adaptive_cli_problem(*common, None, 64, 1e-2, "batch", mean_samples_per_pixel=32) is None
