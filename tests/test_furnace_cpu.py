"""The furnace closed forms of tests/furnace_ref.py pinned to the bit-exact fp64 oracle (oracle/pt_oracle.c):
what makes them a trustworthy reference for the GPU kernels (tests/test_gpu_furnace.py).

* without roulette: every pixel is the closed form, bit for bit in the oracle's operation order and to a few
  ulps as E sum rho^d; the ray count is W H S^2 sum N^d; the hit index is the furnace's index in World order;
* N = 1 with roulette: every sample lies in the admissible set {V(k)} at the k its ray count gives, and the
  histogram of k follows the law of k (fixed-seed chi-square);
* N > 1 with roulette: the sample mean and the mean ray count are within 5 sigma of the closed forms."""
import numpy as np
import pytest

import furnace_ref as fr
from oracle import oracle
from pytracer_b200.flatten import flatten_world
from pytracer_b200.params import make_params
from pytracer_b200.pcg import PCG

NO_RR = 10 ** 6  # rr_limit beyond any depth: no roulette


def _ulps(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b)) / np.spacing(np.abs(np.asarray(b)))))


@pytest.mark.parametrize("N, D", [(1, 8), (2, 6), (3, 5), (40, 2), (1100, 1), (3, 0), (1, 1022)])
def test_closed_form_agrees_with_the_oracle_order(N, D):
    for name in fr.FURNACES:
        _, _, _, rho, E = fr.furnace(name)
        a, b = fr.oracle_value(E, rho, N, D), fr.value(E, rho, D)
        # each level rounds a product, N - 1 additions, the 1/N weight, a scaling and an addition: at most
        # N + 3 roundings of u = 2^-53 per level, and a relative error of k u is at most k ulps
        assert _ulps(a, b) <= (D + 1) * (N + 3), (name, a, b)


CASES = [  # (furnace, decoy spheres, decoy planes, W, H, S, N, D)
    ("diffuse", 0, 0, 5, 3, 2, 2, 4),
    ("diffuse", 3, 2, 4, 3, 3, 1, 8),
    ("mirror", 2, 1, 5, 3, 2, 3, 3),
    ("ellipsoid", 5, 3, 3, 2, 2, 2, 5),
    ("checkered", 1, 4, 3, 2, 1, 3, 0),
    ("image", 4, 0, 3, 2, 2, 2, 3),
    ("black", 2, 2, 3, 2, 2, 5, 4),
    ("diffuse", 40, 1, 2, 2, 1, 40, 2),
    ("mirror", 0, 0, 2, 1, 1, 1100, 1),
    ("ellipsoid", 0, 1, 2, 1, 1, 1, 1022),
    ("diffuse", 2, 1, 3, 2, 2, 3, -1),
]


@pytest.mark.parametrize("name, ns, npl, W, H, S, N, D", CASES, ids=[f"{c[0]}-{c[1]}s{c[2]}p-S{c[5]}-N{c[6]}-D{c[7]}" for c in CASES])
def test_oracle_render_is_the_closed_form(name, ns, npl, W, H, S, N, D):
    world, idx, cam, rho, E = fr.furnace(name, ns, npl)
    p = make_params(W, H, cam, "pathtracing", S, num_of_rays=N, max_depth=D, rr_limit=NO_RR,
                    aa_pcg=PCG(42, 54), pt_pcg=PCG(45, 54))
    r = oracle.render(flatten_world(world), p)
    want = fr.oracle_pixel(fr.oracle_value(E, rho, N, D), S)
    assert np.array_equal(r["rgb"], np.broadcast_to(want, r["rgb"].shape)), (r["rgb"][0, 0], want)
    if D >= 0:
        assert _ulps(want, fr.value(E, rho, D)) <= (D + 1) * (N + 3) + S * S + 1
    spp = max(S, 1) ** 2
    assert r["samples"] == W * H * spp
    assert r["rays_closest"] == W * H * spp * fr.rays_per_sample(N, D, rho)
    assert (r["hit_index"] == (idx if D >= 0 else -1)).all()


@pytest.mark.parametrize("name", ["diffuse", "image", "black"])
@pytest.mark.parametrize("d0", [0, 1, 3, 6])
def test_oracle_trace_rays_from_depth_d0(name, d0):
    world, _, _, rho, E = fr.furnace(name, 3, 1)
    rays = fr.inside_rays(name, 16)
    N, D = 2, 5
    p = make_params(1, 1, fr.furnace_camera("sphere"), "pathtracing", num_of_rays=N, max_depth=D, rr_limit=NO_RR)
    out, _, counters = oracle.trace_rays(flatten_world(world), p, rays, depth=np.full(16, d0, np.int32))
    assert np.array_equal(out, np.broadcast_to(fr.oracle_value(E, rho, N, D, d0), out.shape))
    assert int(counters[0]) == 16 * (fr.rays_per_sample(N, D - d0, rho) if D >= d0 else 0)


def oracle_samples(name, N, D, R, n, seed=9):
    """Per-sample values and ray counts of n rays from the camera position, one oracle call per ray."""
    world, _, _, rho, E = fr.furnace(name, 2, 1)
    fs = flatten_world(world)
    p = make_params(1, 1, fr.furnace_camera("sphere"), "pathtracing", num_of_rays=N, max_depth=D, rr_limit=R)
    rays = fr.inside_rays(name, n, seed)
    st = PCG(seed, 11)
    state = (st.state, st.inc)
    vals, counts = np.zeros((n, 3)), np.zeros(n, np.int64)
    for i in range(n):
        out, state, c = oracle.trace_rays(fs, p, rays[i:i + 1], pcg_state_inc=state)
        vals[i], counts[i] = out[0], int(c[0])
    return vals, counts, rho, E


@pytest.mark.parametrize("name, D, R", [("diffuse", 12, 2), ("mirror", 30, 0), ("ellipsoid", 30, 0), ("checkered", 12, 2)])
def test_oracle_roulette_n1_values_and_law(name, D, R):
    vals, counts, rho, E = oracle_samples(name, 1, D, R, 3000)
    k = counts - 1
    assert (k >= R).all() and (k <= D).all(), (k.min(), k.max())
    exact = fr.oracle_values_by_k(E, rho, R, D)
    assert np.array_equal(vals, exact[k])
    assert _ulps(exact, fr.values_by_k(E, rho, R, D)) <= 8 * (D + 1)
    pv = fr.chi2_pvalue(k, fr.law_of_k(rho, R, D))
    print(f"\n{name} D = {D} R = {R}: chi-square p = {pv:.4f}")
    assert pv >= 1e-6


@pytest.mark.parametrize("name", ["diffuse", "mirror"])
def test_oracle_roulette_many_rays_is_unbiased(name):
    N, D, R = 3, 5, 2
    vals, counts, rho, E = oracle_samples(name, N, D, R, 1500)
    n = vals.shape[0]
    sig_v = vals.std(0, ddof=1) / np.sqrt(n)
    sig_r = counts.std(ddof=1) / np.sqrt(n)
    assert (np.abs(vals.mean(0) - fr.value(E, rho, D)) <= 5 * sig_v).all(), (vals.mean(0), fr.value(E, rho, D), sig_v)
    assert abs(counts.mean() - fr.mean_rays(N, rho, R, D)) <= 5 * sig_r, (counts.mean(), fr.mean_rays(N, rho, R, D))


def test_law_of_k_and_mean_rays_are_consistent():
    for name in ("diffuse", "mirror", "black"):
        _, _, _, rho, E = fr.furnace(name)
        for R, D in ((2, 12), (0, 30), (5, 5), (7, 3)):
            law = fr.law_of_k(rho, R, D)
            assert abs(law.sum() - 1.0) < 1e-12
            if max(rho) > 0:  # N = 1: E[rays] = sum_k (k + 1) P(k); E[V(k)] = the unbiased value
                assert abs(fr.mean_rays(1, rho, R, D) - float((np.arange(D + 1) + 1) @ law)) < 1e-9
                assert np.allclose(law @ fr.values_by_k(E, rho, R, D), fr.value(E, rho, D), rtol=1e-12)
