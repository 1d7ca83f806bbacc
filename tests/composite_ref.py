"""float64 reference and error bound for the averaged full-resolution maps (src/body.py:54-68) that the device computes
from the stride-8 net outputs: the materialised planes of opb_body_maps and, bit for bit the same values, the composite
samples of the fused peak and PAF kernels (csrc/composite.cuh).

Per axis and scale the x8 cubic upsample, the crop and the resize to the frame are one banded operator A (the float64
product of O.composite_upsample_matrix); the averaged map of channel c is

    ref[c] = sum_s (1/S) A_y,s @ V_s[:, :, c] @ A_x,s^T.

Error bound.  The device evaluates, per output element (y, x) and with u = 2^-24 (float32 unit roundoff):
  - x pass: t_k = fmaf chain over the 6 column taps of scale s, starting from 0 -> 6 roundings;
  - y pass: one fmaf chain over all S scales and their 6 row taps -> 6 S roundings (the strip-blocked pass of the
    materialising kernel adds zero-weight taps, which are exact no-ops for finite inputs);
  - weights: the column and row weights are the float64 entries of A rounded once to float32 (one rounding each), and
    the row weights are then divided by S in float32 (one more rounding, exact when S is a power of two).
Each product w_y w_x v of the exact sum therefore reaches the result multiplied by a product of at most
n = 6 + 6 S + 3 factors (1 + d_i), |d_i| <= u, and the standard bound gives

    |device - ref| <= gamma_n * sum_s sum_{k,j} |w_y,s,k / S| |w_x,s,j| |V_s[k, j]|,   gamma_n = n u / (1 - n u).

For n u <= 1e-2 gamma_n <= 1.0102 n u, so c = 1.02 (6 S + 9) covers it together with the float64 rounding of the
reference itself (about 1e-15 relative).  Relative rounding errors hold for normal numbers only: in the subnormal range
(the tails of a Gaussian bump) a rounding errs by up to 2^-150 absolute, so the bound adds c 2^-149.  The bound is per
element and scales with the values that enter that element, so it stays tight inside a window of large dynamic range and does not let a wrong tap hide behind another element's
magnitude.
"""
import numpy as np

from oracle import openpose_oracle as O

U = 2.0 ** -24


def bound_factor(n_scales):
    """c of the per-element bound c * 2^-24 * sum |w_y||w_x||v| (module docstring)."""
    return 1.02 * (6 * n_scales + 9)


def axis_operators(H, W, dims):
    """dims: per scale (h, w, ho, wo) -> per scale (A_y (H, ho), A_x (W, wo)) float64."""
    return [(O.composite_upsample_matrix(ho, h, H), O.composite_upsample_matrix(wo, w, W)) for h, w, ho, wo in dims]


def reference(nets, ops):
    """nets: per scale (ho, wo, C) net outputs; ops: axis_operators.  Returns (ref, mag), both (C, H, W) float64:
    the averaged map and sum_s sum |w_y / S||w_x||v|."""
    S = len(nets)
    ref = mag = 0.0
    for v, (ay, ax) in zip(nets, ops):
        v = np.asarray(v, dtype=np.float64).transpose(2, 0, 1)                     # (C, ho, wo)
        ref = ref + np.matmul(np.matmul(ay, v), ax.T) / S
        mag = mag + np.matmul(np.matmul(np.abs(ay), np.abs(v)), np.abs(ax).T) / S
    return ref, mag


def excess(planes, nets, ops):
    """max over elements of |planes - ref| / bound (<= 1 passes).  planes: (C, H, W) float32 device maps."""
    ref, mag = reference(nets, ops)
    err = np.abs(np.asarray(planes, dtype=np.float64) - ref)
    bound = bound_factor(len(nets)) * (U * mag + 2.0 ** -149)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / bound)
    return float(r.max())


def assert_within_bound(planes, nets, ops, what=""):
    e = excess(planes, nets, ops)
    assert e <= 1.0, "%s: device maps exceed the float64 bound by %.3g x" % (what, e)
    return e


# ---- a float32 stand-in of the device arithmetic (CPU tests of the bound) -----------------------------------------
def taps_of(A):
    """6-tap form of a banded operator: (first index, float32 weights (n, 6)), as net.cu::composite_taps builds it."""
    n = A.shape[0]
    first = np.zeros(n, np.int64)
    w6 = np.zeros((n, 6), np.float32)
    for o in range(n):
        nz = np.nonzero(A[o])[0]
        lo, hi = nz[0], nz[-1]
        assert hi - lo < 6
        first[o] = lo
        w6[o, :hi - lo + 1] = A[o, lo:hi + 1].astype(np.float32)
    return first, w6


def fmaf(a, b, c):
    """float32 fused multiply-add: the product of two float32 values is exact in float64, one rounding per step is
    emulated by rounding the float64 sum to float32 (double rounding may differ from a true fmaf in the last bit)."""
    f64 = np.float64
    return (np.asarray(a, f64) * np.asarray(b, f64) + np.asarray(c, f64)).astype(np.float32)


def standin(nets, ops, mutate=None):
    """The device chains in float32: x pass per scale, then one y chain over all scales, 1/S folded into the row weights.
    nets: per scale (ho, wo, C).  mutate(kind, s, table) may edit a scale's tables: kind 'x' / 'y' (first, w6) or
    'fold' (the divisor) before they are used, or 'row' (a (H, 6) row-index table) for a read from another row.
    Returns (C, H, W) float32."""
    S = len(nets)
    H, W = ops[0][0].shape[0], ops[0][1].shape[0]
    C = nets[0].shape[2]
    acc = np.zeros((C, H, W), np.float32)
    for s, (v, (ay, ax)) in enumerate(zip(nets, ops)):
        v = np.asarray(v, dtype=np.float32).transpose(2, 0, 1)                    # (C, ho, wo)
        ho, wo = v.shape[1:]
        fx, wx = taps_of(ax)
        fy, wy = taps_of(ay)
        div = np.float32(S)
        if mutate:
            fx, wx = mutate("x", s, (fx, wx))
            fy, wy = mutate("y", s, (fy, wy))
            div = mutate("fold", s, div)
        wy = (wy / div).astype(np.float32)
        rows = np.minimum(fy[:, None] + np.arange(6)[None, :], ho - 1)            # (H, 6)
        if mutate:
            rows = mutate("row", s, rows)
        cols = np.minimum(fx[:, None] + np.arange(6)[None, :], wo - 1)            # (W, 6)
        t = np.zeros((C, ho, W), np.float32)                                      # x pass
        for j in range(6):
            t = fmaf(wx[None, None, :, j], v[:, :, cols[:, j]], t)
        for k in range(6):                                                        # y pass, continues over the scales
            acc = fmaf(wy[None, :, k, None], t[:, rows[:, k], :], acc)
    return acc
