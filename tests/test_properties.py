"""Size-independent properties of the restated third-party arithmetic and of the host helpers, on random inputs
(hypothesis) -- and, where /root/reference exists, random-input agreement of the host helpers with the reference's."""
import math

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from oracle import openpose_oracle as O
from oracle import reference_loader as RL
from pytorch_openpose_b200 import util

live = pytest.mark.skipif(not RL.available(), reason="needs a checkout of the original project (set OPENPOSE_REFERENCE_ROOT)")


@settings(max_examples=40, deadline=None)
@given(src=st.integers(4, 400), f=st.floats(0.1, 4.0))
def test_cubic_taps_are_a_partition_of_unity(src, f):
    dst = max(1, O.resize_dsize(src, f))
    first, coef = O.cubic_taps(src, dst, 1.0 / f)
    assert len(first) == dst and np.asarray(coef).shape == (dst, 4)
    assert np.abs(np.asarray(coef, dtype=np.float64).sum(1) - 1).max() < 1e-6
    assert np.all(np.diff(first) >= 0)                           # monotone footprints


@settings(max_examples=25, deadline=None)
@given(n_net=st.integers(2, 40), crop=st.integers(0, 7), f=st.floats(0.5, 9.0))
def test_composite_upsample_preserves_constants_and_linearity(n_net, crop, f):
    """x8 cubic, crop of the padding, cubic resize: every row of the composite operator sums to 1, it has at most 6
    non-zeros, and it is linear (what lets the device apply it as one banded pass per axis)."""
    n_resized = 8 * n_net - crop
    n_orig = max(1, int(round(n_resized * f / 4)))
    M = O.composite_upsample_matrix(n_net, n_resized, n_orig)
    assert M.shape == (n_orig, n_net)
    assert np.abs(M.sum(1) - 1).max() < 1e-5
    assert (np.abs(M) > 0).sum(1).max() <= 6
    rng = np.random.default_rng(n_net * 131 + crop)
    a, b = rng.standard_normal(n_net), rng.standard_normal(n_net)
    assert np.allclose(M @ (2 * a - 3 * b), 2 * (M @ a) - 3 * (M @ b), atol=1e-9)


@settings(max_examples=15, deadline=None)
@given(h=st.integers(1, 60), w=st.integers(1, 60), seed=st.integers(0, 10 ** 6))
def test_gaussian_is_mass_preserving_symmetric_and_scipy_exact(h, w, seed):
    from scipy.ndimage import gaussian_filter
    m = np.random.default_rng(seed).random((h, w)).astype(np.float32).astype(np.float64)
    g = O.gaussian_sigma3(m)
    assert np.array_equal(g, gaussian_filter(m, sigma=3))       # bit-exact at every size, incl. maps smaller than the radius
    assert abs(g.sum() - m.sum()) <= 1e-9 * max(1.0, abs(m.sum()))   # reflect border keeps the mass
    assert np.array_equal(O.gaussian_sigma3(m[::-1, ::-1])[::-1, ::-1], g)


@settings(max_examples=30, deadline=None)
@given(h=st.integers(1, 2000), w=st.integers(1, 4000), s=st.sampled_from([0.5, 1.0, 1.5, 2.0]))
def test_scale_plan_matches_cv2_sizes(h, w, s):
    """dsize = round-half-even(size * multiplier) like cv2.resize(fx, fy); padded sizes are multiples of 8."""
    import cv2
    (p,) = O.scale_plan(h, w, (s,))
    if p["h"] < 1 or p["w"] < 1 or h * w > 4_000_000:
        return
    if h * w <= 40_000:                                          # check against cv2 itself on small frames
        out = cv2.resize(np.zeros((h, w, 3), np.uint8), (0, 0), fx=p["mult"], fy=p["mult"], interpolation=cv2.INTER_CUBIC)
        assert out.shape[:2] == (p["h"], p["w"])
    assert p["hp"] % 8 == 0 and p["wp"] % 8 == 0 and 0 <= p["hp"] - p["h"] < 8 and 0 <= p["wp"] - p["w"] < 8


@live
@settings(max_examples=60, deadline=None)
@given(seed=st.integers(0, 10 ** 6), people=st.integers(0, 4))
def test_hand_detect_matches_reference_on_random_poses(seed, people):
    ns = RL.load()
    rng = np.random.default_rng(seed)
    H, W = int(rng.integers(60, 800)), int(rng.integers(60, 1300))
    cand = np.column_stack([rng.uniform(-20, W + 20, 18 * max(people, 1)), rng.uniform(-20, H + 20, 18 * max(people, 1)),
                            rng.random(18 * max(people, 1)), np.arange(18 * max(people, 1))])
    subset = -np.ones((people, 20))
    for p in range(people):
        for j in range(18):
            if rng.random() > 0.25:
                subset[p, j] = p * 18 + j
    img = np.zeros((H, W, 3), np.uint8)
    ref = ns.util.handDetect(cand, subset, img)
    assert util.handDetect(cand, subset, img) == ref
    assert O.hand_detect(cand, subset, H, W) == ref
    for x, y, w_, _ in ref:                                      # boxes stay inside the frame
        assert 0 <= x and 0 <= y and x + w_ <= W and y + w_ <= H


@live
@settings(max_examples=30, deadline=None)
@given(h=st.integers(1, 50), w=st.integers(1, 50), stride=st.sampled_from([4, 8, 16]), seed=st.integers(0, 999))
def test_pad_and_npmax_match_reference(h, w, stride, seed):
    ns = RL.load()
    img = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    a, pa = util.padRightDownCorner(img, stride, 128)
    b, pb = ns.util.padRightDownCorner(img, stride, 128)
    assert np.array_equal(a, b) and list(pa) == list(pb)
    m = np.random.default_rng(seed + 1).integers(0, 5, (h, w)).astype(np.float64)     # many ties
    assert tuple(util.npmax(m)) == tuple(int(v) for v in ns.util.npmax(m))
