"""The error map against exact host references.

1. SE^2 of every ERR instantiation (k_pt_warp with shapes in the SMALL tables, in shared or in global memory and
   every accumulator; k_pt_warp_bvh) against the fp64 batch estimator of DESIGN.md §5.5, evaluated on the
   per-sample values that S^2 partitioned renders give (a render with part_mode RT_PART_SPP, part_count S^2 and
   part_rank r traces stratum r of every pixel with the sample index, jitter and PCG stream of the full render,
   so S^2 * part_r is sample r).  Every batch layout that groups the samples differently must fail the same
   bound, which pins the task size G the launcher chose.
2. rt_render_adaptive's passes replayed on the host (tests/util.py replay_adaptive) from single-pass renders whose
   PCG states are those of pass p, against one multi-pass call."""
import numpy as np
import pytest

from pytracer_b200 import _abi, scenes
from pytracer_b200.device import DeviceScene
from pytracer_b200.flatten import flatten_world
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG, lcg_advance
from pytracer_b200.scene import World
from util import batch_se2, demo_flat, replay_adaptive, same_partition

pytestmark = pytest.mark.gpu

W, H = 47, 29  # 1 363 pixels: no multiple of 2, 3, 4 or 8, so the last task of every layout is partial
DEMO = dict(num_of_rays=10, max_depth=3, rr_limit=3)
SPHERES = dict(num_of_rays=4, max_depth=3, rr_limit=2)

# (scene, accel, S, path-tracer parameters, G): G follows from the sizing in launch_pt_warp_impl (L = S^2 samples
# per pixel: G = 1 for L >= 32, else ceil(32 / L) up to 8, and for tables outside the SMALL kernel at most 32 / L)
# and launch_pt_warp_bvh (ceil(32 / L) up to 8).  Accumulators the launcher picks (checked once on a B200 with a
# printf in the launchers): demo.txt (SMALL) G = 8, 4 ACC_SEG (the ACC_LANES columns would cost a resident block),
# G = 2 ACC_LANES, G = 1 ACC_REG; 37 spheres (shapes in shared memory) G = 8, 3, 2 ACC_LANES, G = 1 ACC_REG, and
# ACC_SEG at depth 7 (the deeper work stack leaves no room for the columns); 1 400 spheres (global memory) ACC_LANES.
CASES = (
    [("demo", "none", S, DEMO, G) for S, G in ((2, 8), (3, 4), (4, 2), (5, 2), (6, 1), (8, 1))]
    + [("spheres37", "none", S, SPHERES, G) for S, G in ((2, 8), (3, 3), (4, 2), (5, 1), (8, 1))]
    + [("spheres37", "none", 2, dict(SPHERES, max_depth=7), 8)]
    + [("spheres1400", "none", S, SPHERES, G) for S, G in ((3, 3), (4, 2))]  # shape tables > 64 KB: global memory
    + [("spheres37", "bvh", S, SPHERES, G) for S, G in ((2, 8), (3, 4), (4, 2), (5, 2), (6, 1))]
)
CANDIDATE_BPP = (4, 8, 10, 16, 32)  # 32 / G for G = 8, 4, 3, 2, 1

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


def _wrong_layouts(L, bpp):
    """Batch labels of every candidate layout that partitions the L samples differently from s mod bpp: the
    other 32 / G, and contiguous blocks s // n with as many batches as the kernel's layout.  (At S = 2 every
    candidate gives one-sample batches, as the kernel does: there is nothing to tell apart.)"""
    true = np.arange(L) % bpp
    n = -(-L // min(L, bpp))
    cands = [(f"bpp {c}", np.arange(L) % c) for c in CANDIDATE_BPP if c != bpp] + [(f"blocks of {n}", np.arange(L) // n)]
    out = []
    for name, lab in cands:
        if not same_partition(lab, true) and not any(same_partition(lab, o) for _, o in out):
            out.append((name, lab))
    return out


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_error_map_equals_the_fp64_batch_estimator(case):
    name, accel, S, kw, G = case
    sc, cam = _scene(name)
    L, bpp = S * S, 32 // G
    mk = lambda **extra: make_params(W, H, cam, algorithm="pathtracing", samples_per_side=S, aa_pcg=PCG(42, 54),
                                     pt_pcg=PCG(45, 54), accel=accel, **kw, **extra)
    rgb, _, st = sc.render(mk())
    mean, err, samples, ast = sc.render_adaptive(mk(), 0.0, 1)
    assert np.array_equal(mean, rgb)
    assert (samples == L).all() and ast["passes"] == 1 and ast["overflow"] == 0 and st["overflow"] == 0
    parts, rays = [], 0
    for r in range(L):
        img, _, pst = sc.render(mk(part_mode=_abi.RT_PART_SPP, part_count=L, part_rank=r))
        assert pst["overflow"] == 0
        parts.append(img.astype(np.float64))
        rays += pst["rays_closest"]
    assert ast["rays_closest"] == st["rays_closest"] == rays
    x = np.stack(parts, -1) * L                                    # [H][W][3][L]: sample s of every value
    m = mean.astype(np.float64)
    recon = np.stack(parts, -1).sum(-1)
    keep = (np.abs(recon - m) <= 2e-5 * np.abs(m) + 1e-7).all(-1)  # pixels whose samples the partitions reproduce
    dropped = int((~keep).sum())
    assert dropped <= max(2, 0.001 * W * H), dropped

    e2 = err.astype(np.float64) ** 2
    se2, bound = batch_se2(x, bpp, bound=True)
    ratio = np.abs(e2 - se2)[keep] / np.where(bound[keep] > 0, bound[keep], np.inf)
    worst = np.unravel_index(np.argmax(np.where(keep[..., None], np.abs(e2 - se2) - bound, -np.inf)), e2.shape)
    assert (np.abs(e2 - se2) <= bound)[keep].all(), (worst, x[worst], err[worst], mean[worst], se2[worst], bound[worst])
    flat = (x == x[..., :1]).all(-1)                               # every sample the same: no spread to report
    assert (err[flat] <= 1e-6 * np.abs(mean[flat])).all()

    # the same comparison with any other batch layout fails: the bound is tight enough to see the layout
    noisy = keep[..., None] & (se2 > (1e-3 * np.maximum(np.abs(m), 1e-6)) ** 2)
    assert noisy.sum() >= 100, int(noisy.sum())
    fails = []
    for lname, labels in _wrong_layouts(L, bpp):
        s2, b2 = batch_se2(x, labels, bound=True)
        frac = float((np.abs(e2 - s2) > b2)[noisy].mean())
        fails.append(f"{lname} {frac:.3f}")
        assert frac >= 0.9, (lname, frac)
    passing = [c for c in CANDIDATE_BPP if same_partition(np.arange(L) % c, np.arange(L) % bpp)]
    print(f"\n{_case_id(case)}: G = {G} (bpp {bpp}; candidate bpp consistent with the map: {passing}), "
          f"{dropped} pixels dropped by the reconstruction filter, {int(flat.sum())} values without spread, "
          f"largest |err^2 - SE^2_ref| / bound {ratio.max():.3f}; {int(noisy.sum())} noisy values fail other layouts: "
          f"{', '.join(fails) or 'none differs'}")


def test_error_map_of_an_empty_world_is_the_background():
    world = World()
    _, cam = demo_flat()
    sc = DeviceScene(flatten_world(world))
    bg = (0.7, 0.5, 1.0)
    p = make_params(W, H, cam, algorithm="pathtracing", samples_per_side=4, background=bg, aa_pcg=PCG(42, 54),
                    pt_pcg=PCG(45, 54), **DEMO)
    mean, err, samples, st = sc.render_adaptive(p, 0.0, 1)
    want = np.broadcast_to(np.array(bg, dtype=np.float32), mean.shape)
    assert np.array_equal(mean, want) and (err <= 1e-6 * want).all() and (samples == 16).all()
    mean, err, samples, st = sc.render_adaptive(p, 0.01, 4)
    assert st["passes"] == 1 and st["pixels_in_pass"] == [W * H] and (samples == 16).all() and np.array_equal(mean, want)


def _pass_params(w, h, cam, S, pas, **kw):
    """Parameters of pass `pas` of rt_render_adaptive: the jitter state advanced by pas * 2 * W * H * S^2
    draws, the path-tracing state by pas steps."""
    p = make_params(w, h, cam, algorithm="pathtracing", samples_per_side=S, aa_pcg=PCG(11, 3), pt_pcg=PCG(77, 5), **DEMO, **kw)
    p.aa_state = lcg_advance(p.aa_state, p.aa_inc, pas * 2 * w * h * S * S)
    p.pt_state = lcg_advance(p.pt_state, p.pt_inc, pas)
    return p


REPLAYS = [  # (w, h, S, target, floor, max_passes)
    (1024, 576, 8, 0.03, 1e-2, 4),  # pass 0 compacts 288 tiles of 2 048 entries: the carry loop of k_adaptive_offsets
    (97, 61, 8, 0.03, 0.3, 4),      # partial tiles; the floor decides many dark pixels
    (97, 61, 8, float("inf"), 1e3, 4),  # no pixel misses the target: one pass
    (1, 1, 8, 0.001, 1e-2, 3),
    (33, 1, 8, 0.02, 1e-2, 3),
    (160, 120, 4, 0.03, 1e-2, 4),   # G = 2: later passes pair listed pixels, so their sums round differently
]


@pytest.mark.parametrize("w, h, S, target, floor, max_passes", REPLAYS,
                         ids=[f"{w}x{h}-S{S}-target{t:g}-floor{f:g}" for w, h, S, t, f, _ in REPLAYS])
def test_adaptive_passes_equal_the_host_replay(w, h, S, target, floor, max_passes):
    sc, cam = _scene("demo")
    means, errs = [], []
    for pas in range(max_passes):
        m, e, _, st = sc.render_adaptive(_pass_params(w, h, cam, S, pas), 0.0, 1)
        means.append(m)
        errs.append(e)
    # at S = 8 a task is one pixel and a listed pixel is traced as in the full frame, bit for bit; at S = 4 a task
    # pairs pixels of the list, so the pass values of later passes round differently
    exact = S * S >= 32
    r = replay_adaptive(np.stack(means), np.stack(errs), target, floor, max_passes)
    mean, err, samples, st = sc.render_adaptive(_pass_params(w, h, cam, S, 0), target, max_passes, error_floor=floor)
    amb = r["ambiguous"]
    ok = ~amb
    n_amb = int(amb.sum())
    print(f"\n{w}x{h} S = {S}: passes {st['passes']}, pixels per pass {st['pixels_in_pass']} (replay {r['pixels_in_pass']}), "
          f"{n_amb} ambiguous pixels, {int((r['passes'] != samples // (S * S))[ok].sum())} disagreeing")
    assert n_amb <= max(3, 1e-4 * w * h), n_amb
    assert np.array_equal(samples[ok], (r["passes"] * S * S)[ok])
    # the counters, with the kernel's own decision where the replay cannot tell
    P = np.where(amb, samples // (S * S), r["passes"])
    assert st["pixels_in_pass"] == [int((P > p).sum()) for p in range(int(P.max()))][:16]
    assert st["passes"] == int(P.max()) and st["samples"] == int(P.sum()) * S * S and st["overflow"] == 0
    if exact:
        assert np.array_equal(mean[ok], r["mean"][ok])
        assert np.allclose(err[ok], r["err"][ok], rtol=1e-6, atol=0)
    else:
        assert np.allclose(mean[ok], r["mean"][ok], rtol=1e-5, atol=1e-7)
        rel = np.abs(err[ok] - r["err"][ok]) / np.maximum(r["err"][ok], 1e-7)
        print(f"S = {S}: err against the replay: largest relative difference {rel.max():.2e}")
        assert np.allclose(err[ok], r["err"][ok], rtol=1e-5, atol=1e-7)
    if not np.isfinite(target):
        assert st["passes"] == 1 and (samples == S * S).all()
