"""The paired-strata error estimator (RT_ERR_EST_PAIRED) against exact host references, as test_gpu_error_map.py
checks the batch estimator.

1. SE^2 of every ERR instantiation against the fp64 paired estimator (tests/paired_ref.py) evaluated on the
   per-sample values that S^2 renders partitioned with RT_PART_SPP give (S^2 * part_r is sample r), within a
   rounding bound derived from the fp32 batch sums.  The batch estimator must fail that bound, so the mode switched.
2. rt_render_adaptive's passes with the paired estimator replayed on the host (tests/util.py replay_adaptive).
3. The refusals of the C-ABI and the `render --error-estimator paired` command."""
import numpy as np
import pytest

from paired_ref import paired_se2
from pytracer_b200 import _abi, _native, scenes
from pytracer_b200.device import DeviceScene
from pytracer_b200.flatten import flatten_world
from pytracer_b200.hdrimage import HdrImage
from pytracer_b200.imagetracer import CudaImageTracer
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG, lcg_advance
from pytracer_b200.render import PathTracer
from pytracer_b200.scene import World
from util import batch_se2, demo_flat, replay_adaptive

pytestmark = pytest.mark.gpu

W, H = 47, 29  # no multiple of 2 or 8: the last task of every layout is partial
DEMO = dict(num_of_rays=10, max_depth=3, rr_limit=3)
SPHERES = dict(num_of_rays=4, max_depth=3, rr_limit=2)

# (scene, accel, S, path-tracer parameters, G), as in test_gpu_error_map.py.  An even S gives L = 4 (G = 8), 16
# (G = 2) or L >= 32 (G = 1): G = 4 and 3 need L in 5 .. 10, which only odd S reach.  Accumulators: demo.txt
# (SMALL) G = 8 ACC_SEG, G = 2 ACC_LANES, G = 1 ACC_REG; 37 spheres (shapes in shared memory) G = 8, 2 ACC_LANES,
# G = 1 ACC_REG, ACC_SEG at depth 7; 1 400 spheres (global memory) ACC_LANES; k_pt_warp_bvh.
CASES = (
    [("demo", "none", S, DEMO, G) for S, G in ((2, 8), (4, 2), (6, 1), (8, 1), (16, 1))]
    + [("spheres37", "none", S, SPHERES, G) for S, G in ((2, 8), (4, 2), (6, 1))]
    + [("spheres37", "none", 2, dict(SPHERES, max_depth=7), 8)]
    + [("spheres1400", "none", 4, SPHERES, 2)]
    + [("spheres37", "bvh", S, SPHERES, G) for S, G in ((2, 8), (4, 2), (6, 1))]
)

_scenes = {}


def _scene(name):
    if name not in _scenes:
        if name == "demo":
            fs, cam = demo_flat()
        else:
            rs = scenes.random_spheres_scene(int(name[len("spheres"):]))
            fs, cam = flatten_world(rs.world), rs.camera
        _scenes[name] = (DeviceScene(fs), cam)
    return _scenes[name]


def _case_id(c):
    scene, accel, S, kw, G = c
    return f"{scene}-{accel}-S{S}-depth{kw['max_depth']}-G{G}"


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_paired_error_map_equals_the_fp64_paired_estimator(case):
    name, accel, S, kw, G = case
    sc, cam = _scene(name)
    L, bpp = S * S, 32 // G
    mk = lambda **extra: make_params(W, H, cam, algorithm="pathtracing", samples_per_side=S, aa_pcg=PCG(42, 54),
                                     pt_pcg=PCG(45, 54), accel=accel, **kw, **extra)
    rgb, _, st = sc.render(mk())
    mean, err, samples, ast = sc.render_adaptive(mk(), 0.0, 1, estimator="paired")
    assert np.array_equal(mean, rgb)
    assert (samples == L).all() and ast["passes"] == 1 and ast["overflow"] == 0 and st["overflow"] == 0
    assert (ast["rays_closest"], ast["rays_shadow"], ast["samples"]) == (st["rays_closest"], st["rays_shadow"], st["samples"])
    parts = []
    for r in range(L):
        img, _, pst = sc.render(mk(part_mode=_abi.RT_PART_SPP, part_count=L, part_rank=r))
        assert pst["overflow"] == 0
        parts.append(img.astype(np.float64))
    x = np.stack(parts, -1) * L                                    # [H][W][3][L]: sample s of every value
    m = mean.astype(np.float64)
    keep = (np.abs(np.stack(parts, -1).sum(-1) - m) <= 2e-5 * np.abs(m) + 1e-7).all(-1)  # as test_gpu_error_map.py
    dropped = int((~keep).sum())
    assert dropped <= max(2, 0.001 * W * H), dropped

    e2 = err.astype(np.float64) ** 2
    se2, bound = paired_se2(x, bpp, bound=True)
    ratio = np.abs(e2 - se2)[keep] / np.where(bound[keep] > 0, bound[keep], np.inf)
    worst = np.unravel_index(np.argmax(np.where(keep[..., None], np.abs(e2 - se2) - bound, -np.inf)), e2.shape)
    assert (np.abs(e2 - se2) <= bound)[keep].all(), (worst, x[worst], err[worst], mean[worst], se2[worst], bound[worst])
    flat = (x == x[..., :1]).all(-1)
    assert (err[flat] <= 1e-6 * np.abs(mean[flat])).all()

    # the batch estimator of the same sums fails the paired bound: the kernel really formed the pair differences.
    # At S = 2 the two formulas agree exactly wherever three of the four samples are equal (one outlier c among
    # a, a, a: (c - a)^2 / 16 both), the commonest noisy value there, so the check runs on the values they tell apart.
    noisy = keep[..., None] & (se2 > (1e-3 * np.maximum(np.abs(m), 1e-6)) ** 2)
    batch = batch_se2(x, bpp)
    judged = noisy & (np.abs(batch - se2) > 2.0 * bound) if S == 2 else noisy
    assert judged.sum() >= 100, int(judged.sum())
    frac = float((np.abs(e2 - batch) > bound)[judged].mean())
    assert frac >= 0.9, frac
    print(f"\n{_case_id(case)}: {dropped} pixels dropped by the reconstruction filter, {int(flat.sum())} values without "
          f"spread, largest |err^2 - SE^2_paired| / bound {ratio.max():.3f}; the batch estimator fails the bound on "
          f"{frac:.3f} of {int(judged.sum())} judged values ({int(noisy.sum())} noisy)")


def test_paired_error_map_of_an_empty_world_is_zero():
    _, cam = demo_flat()
    sc = DeviceScene(flatten_world(World()))
    bg = (0.7, 0.5, 1.0)
    p = make_params(W, H, cam, algorithm="pathtracing", samples_per_side=4, background=bg, aa_pcg=PCG(42, 54),
                    pt_pcg=PCG(45, 54), **DEMO)
    want = np.broadcast_to(np.array(bg, dtype=np.float32), (H, W, 3))
    mean, err, samples, st = sc.render_adaptive(p, 0.0, 1, estimator="paired")
    assert np.array_equal(mean, want) and (err <= 1e-6 * want).all() and (samples == 16).all()
    mean, err, samples, st = sc.render_adaptive(p, 0.01, 4, estimator="paired")
    assert st["passes"] == 1 and st["pixels_in_pass"] == [W * H] and (samples == 16).all() and np.array_equal(mean, want)


def _pass_params(w, h, cam, S, pas):
    """Parameters of pass `pas` of rt_render_adaptive (as in test_gpu_error_map.py)."""
    p = make_params(w, h, cam, algorithm="pathtracing", samples_per_side=S, aa_pcg=PCG(11, 3), pt_pcg=PCG(77, 5), **DEMO)
    p.aa_state = lcg_advance(p.aa_state, p.aa_inc, pas * 2 * w * h * S * S)
    p.pt_state = lcg_advance(p.pt_state, p.pt_inc, pas)
    return p


REPLAYS = [  # (w, h, S, target, floor, max_passes)
    (1024, 576, 8, 0.03, 1e-2, 4),  # pass 0 compacts 288 tiles: the carry loop of k_adaptive_offsets
    (97, 61, 8, 0.03, 0.3, 4),      # partial tiles; the floor decides many dark pixels
    (33, 1, 8, 0.02, 1e-2, 3),
    (160, 120, 4, 0.03, 1e-2, 4),   # G = 2: later passes pair listed pixels, so their sums round differently
    (160, 120, 2, 0.05, 1e-2, 4),   # G = 8, two pair differences per pixel
]


@pytest.mark.parametrize("w, h, S, target, floor, max_passes", REPLAYS,
                         ids=[f"{w}x{h}-S{S}-target{t:g}-floor{f:g}" for w, h, S, t, f, _ in REPLAYS])
def test_paired_adaptive_passes_equal_the_host_replay(w, h, S, target, floor, max_passes):
    sc, cam = _scene("demo")
    means, errs = [], []
    for pas in range(max_passes):
        m, e, _, _ = sc.render_adaptive(_pass_params(w, h, cam, S, pas), 0.0, 1, estimator="paired")
        means.append(m)
        errs.append(e)
    r = replay_adaptive(np.stack(means), np.stack(errs), target, floor, max_passes)
    mean, err, samples, st = sc.render_adaptive(_pass_params(w, h, cam, S, 0), target, max_passes, error_floor=floor,
                                                estimator="paired")
    amb = r["ambiguous"]
    ok = ~amb
    n_amb = int(amb.sum())
    print(f"\n{w}x{h} S = {S}: passes {st['passes']}, pixels per pass {st['pixels_in_pass']} (replay {r['pixels_in_pass']}), "
          f"{n_amb} ambiguous pixels")
    assert n_amb <= max(3, 1e-4 * w * h), n_amb
    assert np.array_equal(samples[ok], (r["passes"] * S * S)[ok])
    P = np.where(amb, samples // (S * S), r["passes"])
    assert st["pixels_in_pass"] == [int((P > p).sum()) for p in range(int(P.max()))][:16]
    assert st["passes"] == int(P.max()) and st["samples"] == int(P.sum()) * S * S and st["overflow"] == 0
    if S * S >= 32:  # one-pixel tasks: a listed pixel is traced as in the full frame, bit for bit
        assert np.array_equal(mean[ok], r["mean"][ok])
        assert np.allclose(err[ok], r["err"][ok], rtol=1e-6, atol=0)
    else:
        assert np.allclose(mean[ok], r["mean"][ok], rtol=1e-5, atol=1e-7)
        assert np.allclose(err[ok], r["err"][ok], rtol=1e-5, atol=1e-7)


def test_paired_estimator_refusals():
    sc, cam = _scene("demo")
    for S in (3, 5):  # a stratum without a partner
        with pytest.raises(_native.NativeError) as e:
            sc.render_adaptive(make_params(32, 24, cam, algorithm="pathtracing", samples_per_side=S, **DEMO), 0.0, 1,
                               estimator="paired")
        assert e.value.code == _abi.RT_ERR_INVALID
    for est in (2, -1):
        with pytest.raises(_native.NativeError) as e:
            sc.render_adaptive(make_params(32, 24, cam, algorithm="pathtracing", samples_per_side=4, **DEMO), 0.0, 1,
                               estimator=est)
        assert e.value.code == _abi.RT_ERR_INVALID
    # the default is the batch estimator: one call without the argument equals RT_ERR_EST_BATCH
    p = lambda: make_params(32, 24, cam, algorithm="pathtracing", samples_per_side=4, aa_pcg=PCG(1, 2), pt_pcg=PCG(3, 4), **DEMO)
    a, b = sc.render_adaptive(p(), 0.0, 1), sc.render_adaptive(p(), 0.0, 1, estimator=_abi.RT_ERR_EST_BATCH)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_render_command_writes_the_paired_error_map(tmp_path):
    from click.testing import CliRunner

    from pytracer_b200.hdrimage import read_pfm_image
    from pytracer_b200.main import cli
    from pytracer_b200.scene_text import parse_scene_text
    from test_adaptive_cpu import DEMO_TXT

    scene = tmp_path / "demo.txt"
    scene.write_text(DEMO_TXT)
    out = {k: tmp_path / k for k in ("img.pfm", "img.png", "err.pfm")}
    result = CliRunner().invoke(cli, ["render", "--width", "96", "--height", "72", "--samples-per-pixel", "16",
                                      "--error-estimator", "paired", "--error-output", str(out["err.pfm"]),
                                      "--pfm-output", str(out["img.pfm"]), "--png-output", str(out["img.png"]), str(scene)])
    print(result.output)
    assert result.exit_code == 0, result.output
    parsed = parse_scene_text(DEMO_TXT)
    runs = {}
    for est in ("paired", "batch"):
        image = HdrImage(96, 72)
        res = CudaImageTracer(image, parsed.camera, samples_per_side=4).fire_all_rays_adaptive(
            PathTracer(parsed.world, pcg=PCG(45, 54), num_of_rays=10, max_depth=3), error_estimator=est)
        runs[est] = (image.rgb_array(), res.error)
    with open(out["err.pfm"], "rb") as f:
        err = read_pfm_image(f).rgb_array()
    with open(out["img.pfm"], "rb") as f:
        img = read_pfm_image(f).rgb_array()
    assert np.array_equal(err, runs["paired"][1]) and np.array_equal(img, runs["paired"][0])
    assert np.array_equal(runs["batch"][0], runs["paired"][0]) and not np.array_equal(runs["batch"][1], runs["paired"][1])
