"""Shared helpers of the test-suite: golden fixtures (outputs of the unmodified reference, see
tests/golden/make_golden.py) and scene rebuilding from them."""
import hashlib
import os

import numpy as np

from pytracer_b200 import _abi
from pytracer_b200.flatten import FlatScene
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return np.load(os.path.join(GOLDEN, name))


def sha256_of(a) -> str:
    """Digest of an array's bytes: what a fixture keeps of an image too large to store."""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def camera_from(vec) -> _abi.rt_camera:
    cam = _abi.rt_camera()
    cam.kind, cam.screen_distance, cam.aspect_ratio = int(vec[0]), float(vec[1]), float(vec[2])
    cam.m[:] = [float(v) for v in vec[3:15]]
    return cam


def demo_flat():
    z = golden("demo_scene.npz")
    return FlatScene.from_npz_dict(z), camera_from(z["camera"])


def scene2_flat():
    z = golden("scene2.npz")
    return FlatScene.from_npz_dict(z), camera_from(z["camera"]), camera_from(z["camera_ortho"])


def c1_params(cam, **kw):
    """BASELINE config 1: the reference CLI defaults, 160x120, 1 spp."""
    args = dict(algorithm="pathtracing", samples_per_side=1, num_of_rays=10, max_depth=3, rr_limit=3,
                aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54))
    args.update(kw)
    return make_params(160, 120, cam, **args)


def luminosity(rgb):
    """Color.luminosity, colors.py:59-61, per pixel."""
    return (rgb.max(axis=-1) + rgb.min(axis=-1)) / 2


def mc_agreement(gpu_mean, ref_runs, samples_ratio, n_ref, rel_floor=1e-5):
    """Per-value agreement of a GPU image with K independent oracle runs of the same estimator.

    The north star's bar is "per-pixel means within 3 sigma of the Monte Carlo error"; SURVEY §8(c) adds
    "for >= 99.7 % of pixels", which is the two-sided normal probability of 3 sigma when sigma is KNOWN.
    Here sigma is estimated from K runs, so under the null hypothesis the statistic
        z = (gpu - mean_ref) / (sem_ref * sqrt(1 + samples_ratio))        samples_ratio = n_ref / n_gpu
    follows Student's t with K - 1 degrees of freedom, not a normal: the bound that keeps 99.73 % of the
    values inside is t_crit(K - 1) (3.6 for K = 16), and 3 itself keeps P(|t_{K-1}| < 3) (99.1 % for K = 16).
    Both fractions are returned with their expectations.  The t law needs run means that are close to
    normal: the per-sample distribution of a path tracer is skewed, and with 4 samples per run an ORACLE
    image of 1 024 spp scores 0.9946 / 0.9906 against 24 oracle runs (expected 0.9973 / 0.9936) — with 16
    samples per run it scores 0.9976 / 0.9951 (measured on demo.txt, DESIGN.md §7), so the callers give
    every run at least 16 samples per value.  `rel_floor`, the colour tolerance of the deterministic
    renderers (fp32 against fp64), is granted on top.  Values on which all oracle samples agree (misses,
    emitters seen directly) have no sigma to test against, yet need not be deterministic: if a fraction f of
    the footprint shows something else, all n_ref oracle samples miss it with probability (1 - f)^n_ref,
    which stays above the 3-sigma level 0.0027 up to f = 5.9 / n_ref — so such a value may differ by that
    fraction of the image's value range (the "rule of three" at 3 sigma), and by no more."""
    from scipy import stats

    ref_runs = np.asarray(ref_runs, dtype=np.float64)
    k = ref_runs.shape[0]
    ref_mean = ref_runs.mean(0)
    sem = ref_runs.std(0, ddof=1) / np.sqrt(k) * np.sqrt(1.0 + samples_ratio)
    diff = np.abs(np.asarray(gpu_mean, dtype=np.float64) - ref_mean)
    floor = rel_floor * np.maximum(np.abs(ref_mean), 1e-3)
    # (a spread at the level of fp64 rounding — runs that differ in the last bits of a sum — is no Monte Carlo
    # error to test against: such values count as deterministic)
    noisy = sem > 1e-9 * np.maximum(np.abs(ref_mean), 1e-3)
    crit = float(stats.t.ppf(1.0 - 0.00135, k - 1))
    n = max(1, int(noisy.sum()))
    out = dict(
        k=k, n_noisy=int(noisy.sum()), n_deterministic=int((~noisy).sum()), t_crit=crit,
        frac_3sigma=float((diff[noisy] <= 3.0 * sem[noisy] + floor[noisy]).mean()) if noisy.any() else 1.0,
        expect_3sigma=float(1.0 - 2.0 * stats.t.sf(3.0, k - 1)),
        frac_tcrit=float((diff[noisy] <= crit * sem[noisy] + floor[noisy]).mean()) if noisy.any() else 1.0,
        expect_tcrit=0.9973,
        deterministic_ok=float((diff[~noisy] <= floor[~noisy] + (5.9 / n_ref) * max(1.0, float(np.abs(ref_mean).max()))).mean())
        if (~noisy).any() else 1.0,
        deterministic_exact=float((diff[~noisy] <= floor[~noisy]).mean()) if (~noisy).any() else 1.0,
        worst_z=float((np.maximum(diff[noisy] - floor[noisy], 0.0) / sem[noisy]).max()) if noisy.any() else 0.0,
    )
    # three binomial standard deviations of sampling slack on the expected fractions
    out["bar_3sigma"] = out["expect_3sigma"] - 3.0 * np.sqrt(out["expect_3sigma"] * (1 - out["expect_3sigma"]) / n)
    out["bar_tcrit"] = 0.9973 - 3.0 * np.sqrt(0.9973 * 0.0027 / n)
    return out


def assert_mc_agreement(gpu_mean, ref_runs, samples_ratio, n_ref, what="", rel_floor=1e-5):
    """`n_ref`: oracle samples behind every value (runs x samples per pixel)."""
    r = mc_agreement(gpu_mean, ref_runs, samples_ratio, n_ref, rel_floor)
    print(f"{what}: {r['n_noisy']} noisy values, K = {r['k']}: within 3 sigma {r['frac_3sigma']:.4f} (Student-t expects "
          f"{r['expect_3sigma']:.4f}), within the 99.73 % bound t = {r['t_crit']:.2f}: {r['frac_tcrit']:.4f}, worst z {r['worst_z']:.1f}; "
          f"{r['n_deterministic']} values without oracle variance: {r['deterministic_exact']:.4f} within {rel_floor:g}, "
          f"{r['deterministic_ok']:.4f} within the rule-of-three bound")
    assert r["frac_tcrit"] >= r["bar_tcrit"], (what, r)
    assert r["frac_3sigma"] >= r["bar_3sigma"], (what, r)
    assert r["deterministic_ok"] == 1.0, (what, r)
    return r


def assert_luminance_agreement(gpu_img, ref_runs, what=""):
    """Image-mean luminance within 0.5 % of the oracle's (north star).  Color.luminosity (colors.py:59-61) is
    (max + min) / 2 — not linear in the pixel, so the image mean of a NOISY image is biased (the oracle's own
    image mean of the config-4 scene moves from 0.557 at 1 spp to 0.550 at 9 spp): both sides are therefore
    evaluated on converged pixels — `gpu_img` on the oracle's pixel grid with at least as many samples per
    pixel, the oracle as the mean image of all its runs; its standard error comes from a jackknife over the
    runs.  Where three standard errors exceed 0.5 % (tiny frames) that is the bar, and the message says so."""
    ref_runs = np.asarray(ref_runs, dtype=np.float64)
    k = ref_runs.shape[0]
    total = ref_runs.sum(0)
    lum_ref = luminosity(total / k).mean()
    jack = np.array([luminosity((total - ref_runs[j]) / (k - 1)).mean() for j in range(k)])
    sem = np.sqrt((k - 1) / k * ((jack - jack.mean()) ** 2).sum())
    lum_gpu = luminosity(np.asarray(gpu_img, dtype=np.float64)).mean()
    bar = max(0.005 * lum_ref, 3.0 * sem)
    print(f"{what}: image-mean luminance GPU {lum_gpu:.5f}, oracle {lum_ref:.5f} +- {sem:.5f} "
          f"(difference {abs(lum_gpu / lum_ref - 1) * 100:.3f} %, bar {bar / lum_ref * 100:.2f} %)")
    assert abs(lum_gpu - lum_ref) <= bar, (what, lum_gpu, lum_ref, sem)
    # the linear functional next to it: image-mean RGB, unbiased whatever the sample counts
    rgb_runs = ref_runs.reshape(k, -1, 3).mean(1)
    rgb_ref, rgb_sem = rgb_runs.mean(0), rgb_runs.std(0, ddof=1) / np.sqrt(k)
    rgb_gpu = np.asarray(gpu_img, dtype=np.float64).reshape(-1, 3).mean(0)
    assert (np.abs(rgb_gpu - rgb_ref) <= np.maximum(0.005 * rgb_ref, 3.0 * rgb_sem)).all(), (what, rgb_gpu, rgb_ref, rgb_sem)
