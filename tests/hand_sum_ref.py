"""Host mirror of the certification bound of the hand component choice (csrc/hand.cu, select_cut).

Every component of a map has m <= M values whose magnitudes add up to at most A (M and A of the whole mask).  Any
float64 summation order of m values is within γ_(m-1)·Σ|v| of the exact sum, γ_k = k·u / (1 − k·u), u = 2^-53 (Higham,
Accuracy and Stability of Numerical Algorithms, §4.2); numpy's float32 pairwise sum is within γ_d·Σ|v| with u = 2^-24,
d the most roundings one element passes through in the pairwise tree of any length up to the map's pixel count.  So
the device's float64 sum of a component and numpy's differ by at most

    B = (γ_M(2^-53) + γ') · A / (1 − γ_M(2^-53)),   γ' = γ_M(2^-53) for Hand, γ_d(2^-24) for Batch_hand,

the last factor because A is itself a float64 sum of M magnitudes.  A component is a contender when its device sum is
within 2B of the top one.  The device rounds every step outwards; here the same quantities are evaluated in float64 and
widened by one part in 2^40, far more than the handful of roundings involved."""
import numpy as np


def pairwise_split(n):
    n2 = n // 2
    return n2 - n2 % 8


def pairwise_depth_table(n):
    """d[k] = the most roundings an element passes through in numpy's pairwise sum of k values, for k <= n."""
    d = np.zeros(n + 1, dtype=np.int64)
    for k in range(1, n + 1):
        if k < 8:
            d[k] = k
        elif k <= 128:
            d[k] = k // 8 - 1 + 3 + k % 8
        else:
            k2 = pairwise_split(k)
            d[k] = 1 + max(d[k2], d[k - k2])
    return d


def pairwise_depth_max(n):
    return int(pairwise_depth_table(n).max())


def gamma(k, u):
    return k * u / (1.0 - k * u)


def bound(A, M, f32_depth=0):
    """B above for a map whose mask has M pixels with Σ|v| = A; f32_depth = 0 for Hand (float64 sums)."""
    g = gamma(M, 2.0 ** -53)
    g2 = gamma(f32_depth, 2.0 ** -24) if f32_depth else g
    return (g + g2) * A / (1.0 - g) * (1.0 + 2.0 ** -40)


def warp_atomic_order_sum(raw, mask, rng=None):
    """The float64 sum hand_flatten_kernel forms for one component: 32-lane butterfly sums where a whole warp (32
    columns starting at a multiple of 32) lies in the component, single values elsewhere, added one after another in
    raster order (rng: in a shuffled order, as atomics from different warps may land)."""
    h, w = raw.shape
    parts = []
    for y in range(h):
        for x0 in range(0, w, 32):
            seg, vals = mask[y, x0:x0 + 32], raw[y, x0:x0 + 32].astype(np.float64)
            if len(seg) == 32 and seg.all():
                v = vals.copy()
                for o in (16, 8, 4, 2, 1):
                    v = v + v[np.arange(32) ^ o]
                parts.append(v[0])
            else:
                parts.extend(vals[seg].tolist())
    parts = np.array(parts, dtype=np.float64)
    if rng is not None:
        rng.shuffle(parts)
    return float(np.cumsum(parts)[-1]) if len(parts) else 0.0


def component_sums(m, binary, dtype):
    """Labels (scipy, 8-connectivity) and numpy's sum of every component, as the reference forms them."""
    from scipy import ndimage as ndi
    lab, n = ndi.label(binary, structure=np.ones((3, 3), dtype=int))
    mm = np.asarray(m, dtype=dtype)
    return lab, n, [np.sum(mm[lab == i]) for i in range(1, n + 1)]
