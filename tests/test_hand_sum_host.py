"""CPU checks of the arithmetic behind the hand component choice: the library's pairwise sum is np.sum bit for bit,
and the certification bound (tests/hand_sum_ref.py) holds for every summation order the device can produce while
still leaving ordinary maps without contenders."""
import ctypes

import numpy as np
import pytest

from oracle import openpose_oracle as O
from oracle.make_golden import smooth_noise_maps
from pytorch_openpose_b200 import _lib
from tests import hand_sum_ref as H


def lib_sum(a):
    a = np.ascontiguousarray(a)
    out = ctypes.c_double()
    _lib.check(_lib.lib().opb_debug_pairwise_sum(a.ctypes.data, len(a), int(a.dtype == np.float32), ctypes.byref(out)))
    return a.dtype.type(out.value)


def hard_values(rng, n, dtype):
    """Magnitudes over 1e-30 … 1e4, both signs, exact cancellations and negative zeros."""
    v = rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-30, 4, n)
    k = rng.integers(0, 4)
    if k == 1:                                       # large values that cancel, small ones in between
        big = rng.random(n) < 0.3
        v[big] = 1e4 * rng.choice([-1.0, 1.0], big.sum())
    elif k == 2:
        v[rng.random(n) < 0.2] = -0.0
    elif k == 3:
        v = np.abs(v)
    return v.astype(dtype)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_pairwise_sum_equals_numpy_every_length(dtype):
    rng = np.random.default_rng(1)
    for n in range(1, 1101):
        a = hard_values(rng, n, dtype)
        got, ref = lib_sum(a), np.sum(a)
        assert got.tobytes() == ref.tobytes(), (n, got, ref)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_pairwise_sum_equals_numpy_long_and_masked(dtype):
    rng = np.random.default_rng(2)
    for n in list(rng.integers(1100, 1_000_001, 12)) + [1_000_000, 131072, 129, 128, 127]:
        a = hard_values(rng, int(n), dtype)
        assert lib_sum(a).tobytes() == np.sum(a).tobytes(), n
    m = hard_values(rng, 300 * 300, dtype).reshape(300, 300)       # the reference's raw[lab == i] gather
    sel = m[rng.random((300, 300)) < 0.5]
    assert lib_sum(sel).tobytes() == np.sum(sel).tobytes()


def test_pairwise_sum_signed_zeros_and_empty():
    for dtype in (np.float32, np.float64):
        for n in (1, 3, 8, 9, 200):
            a = np.full(n, -0.0, dtype)
            assert lib_sum(a).tobytes() == np.sum(a).tobytes()
        assert lib_sum(np.zeros(0, dtype)) == 0


def test_pairwise_depth():
    d = H.pairwise_depth_table(2000)
    rng = np.random.default_rng(3)
    for n in (1, 7, 8, 127, 128, 129, 1000, 2000):
        # one element perturbed by its own ulp: its contribution passes through at most d[n] roundings, so the float32
        # sum of values that are all exact in float64 stays within γ_d·Σ|v| of the exact sum
        a = rng.random(n).astype(np.float32)
        exact = np.sum(a.astype(np.float64))
        assert abs(float(np.sum(a)) - exact) <= H.gamma(int(d[:n + 1].max()), 2.0 ** -24) * exact
    assert d[127] == 24 and d[128] == 18 and d[7] == 7


def _assert_within(raw, mask, ref, B, rng):
    orders = [np.cumsum(raw[mask])[-1], np.cumsum(raw[mask][::-1])[-1],
              np.cumsum(rng.permutation(raw[mask]))[-1],
              H.warp_atomic_order_sum(raw, mask), H.warp_atomic_order_sum(raw, mask, rng)]
    for s in orders:
        assert abs(float(s) - float(ref)) <= B


def test_bound_holds_for_device_orders_hand():
    """float64 components whose values span 1e-12 … 1 and cancel: every order the device may add them in stays
    within the bound of np.sum."""
    rng = np.random.default_rng(4)
    worst = 0.0
    for t in range(40):
        h, w = rng.integers(8, 90, 2)
        raw = (rng.choice([-1.0, 1.0], (h, w)) * rng.random((h, w)) * 10.0 ** rng.uniform(-12, 0, (h, w)))
        raw = raw.astype(np.float32).astype(np.float64)
        mask = rng.random((h, w)) < 0.9
        ref = np.sum(raw[mask])
        B = H.bound(np.abs(raw[mask]).sum(), mask.sum())
        _assert_within(raw, mask, ref, B, rng)
        worst = max(worst, max(abs(np.cumsum(rng.permutation(raw[mask]))[-1] - ref) for _ in range(5)) / B)
    assert 0 < worst < 1


def test_bound_holds_for_device_orders_batch_hand():
    """float32 components (numpy sums them in float32, the device in float64), including one-ulp near ties."""
    rng = np.random.default_rng(5)
    for t in range(40):
        h, w = rng.integers(8, 120, 2)
        raw = (rng.random((h, w)) * 10.0 ** rng.uniform(-6, 0, (h, w))).astype(np.float32)
        if t % 2:
            raw[rng.integers(0, h), rng.integers(0, w)] *= -1
        mask = rng.random((h, w)) < 0.95
        ref = np.sum(raw[mask])                               # float32, pairwise
        r64 = raw.astype(np.float64)
        B = H.bound(np.abs(r64[mask]).sum(), mask.sum(), H.pairwise_depth_max(int(h * w)))
        _assert_within(r64, mask, ref, B, rng)


def _no_contenders(maps, binary_of, dtype, f32_depth=0):
    """Per map: the top component's numpy sum exceeds every other one's by more than 4B, so device sums (each within
    B of numpy's) can never bring a second component within 2B of the top: the exact path never runs."""
    checked = 0
    for m in maps:
        binary = binary_of(m)
        if not binary.any():
            continue
        lab, n, sums = H.component_sums(m, binary, dtype)
        vals = np.asarray(m, dtype=np.float64)[binary]
        B = H.bound(np.abs(vals).sum(), int(binary.sum()), f32_depth)
        s = np.sort(np.asarray(sums, dtype=np.float64))[::-1]
        if n > 1:
            assert s[0] - s[1] > 4 * B, (s[0], s[1], B)
            checked += 1
    return checked


def test_ordinary_maps_have_no_contenders():
    """The bound is not vacuous: the golden hand scene and the speckle maps of the stage tests never take the exact
    path, in Hand's float64 and in Batch_hand's float32 setting."""
    hm = smooth_noise_maps(184, 184, 22, 5, 0.03, 21)
    hm[:, :, 3] = -1.0
    speckle = smooth_noise_maps(120, 150, 11, 1.0, 0.06, 41)
    hand = lambda m: O.gaussian_sigma3(m) > O.HAND_THRE
    maps = [hm[:, :, p] for p in range(21)] + [speckle[:, :, p] for p in range(11)]
    assert _no_contenders(maps, hand, np.float64) >= 15
    blurred = O.blur5_fixed_order(hm)
    b32 = [blurred[:, :, p].astype(np.float32) for p in range(21)]
    assert _no_contenders(b32, lambda m: m > np.float32(O.BATCH_HAND_THRE), np.float32,
                          H.pairwise_depth_max(184 * 184)) >= 5
