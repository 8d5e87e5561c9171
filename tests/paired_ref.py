"""fp64 host reference of the paired-strata (collapsed strata) error estimator, RT_ERR_EST_PAIRED.

Imported by the CPU and GPU tests of the estimator; the batch estimator's reference is tests/util.py batch_se2."""
import numpy as np


def paired_se2(x, bpp, bound=False):
    """SE^2 of the pass mean from paired batch sums, in fp64, as DESIGN.md §5.5 documents it (rt_warp.cuh err_store).

    `x`: per-sample values [..., L], the last axis in sample order (stratum ls = row * S + column, so samples 2k
    and 2k + 1 are horizontal neighbours); `bpp` = 32 / G, even.  Sample s goes to batch s mod bpp; with T_b the
    batch sums, group j < min(L, bpp) / 2 forms D_j = T_2j - T_2j+1 and
        SE^2 = sum_j D_j^2 / L^2.
    With `bound=True` also returns how far an fp32 kernel's value may lie from it: every T_b off by at most
    delta_b = 1e-5 sum_{s in b} |x_s| (fp32 sums of the rays of the batch, as batch_se2 takes them), so D_j by
    delta_2j + delta_2j+1, which moves D_j^2 by at most 2 |D_j| delta + delta^2; plus eleven roundings of at most
    2^-24 each of the result: the subtraction (twice, squared), the product, four levels of the butterfly sum of
    at most 16 non-negative terms, 1 / L^2, the scaling, and the square root of the stored SE (twice, squared)."""
    x = np.asarray(x, dtype=np.float64)
    L = x.shape[-1]
    assert L % 2 == 0 and bpp % 2 == 0, (L, bpp)
    b = np.arange(L) % bpp
    groups = min(L, bpp) // 2
    w = np.zeros((L, groups))
    w[np.arange(L), b // 2] = np.where(b % 2 == 0, 1.0, -1.0)
    d = x @ w
    se2 = (d * d).sum(-1) / float(L * L)
    if not bound:
        return se2
    delta = 1e-5 * (np.abs(x) @ np.abs(w))
    return se2, (2.0 * np.abs(d) * delta + delta * delta).sum(-1) / float(L * L) + ((1.0 + 2.0 ** -24) ** 11 - 1.0) * se2
