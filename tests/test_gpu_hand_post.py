"""The hand post-processing kernels (csrc/hand.cu) on crafted maps, through opb_hand_debug_post in all three launch
geometries: Hand on equal-size crops, Hand on a list of crop sides, Batch_hand.  Smoothed planes and labels are checked
against scipy, key points against the oracle, and the component choice on near ties, where the device's atomic sums
alone cannot decide as numpy does.  Every case asserts on oracle-side quantities that it reaches what it is for."""

import numpy as np
import pytest
import torch
from scipy import ndimage as ndi

from oracle import openpose_oracle as O
from oracle.make_golden import smooth_noise_maps
from tests import hand_sum_ref as H

pytestmark = pytest.mark.gpu

EIGHT = np.ones((3, 3), dtype=int)


def post(maps, mode=0, sides=None, flags=0, smoothed=False, labels=False, sums=False):
    """maps: (n_crops, 21, h, w) float32, or for a sides list (n_crops, 21, wmax * wmax) with crop c stored densely
    with width sides[c].  Returns peaks (n_crops, 21, 3) and the requested planes (numpy, at the geometry's pitch)."""
    from pytorch_openpose_b200 import _lib
    from tests import gpu_util as G
    maps = np.ascontiguousarray(maps, dtype=np.float32)
    n = maps.shape[0]
    if sides is None:
        h, w = maps.shape[2:]
        shape = (n, 21, h, w)
    else:
        h = w = 0
        shape = (n, 21, maps.shape[2])
    d = torch.from_numpy(maps).cuda()
    out = {k: torch.zeros(shape, dtype=t, device="cuda") if on else None
           for k, t, on in (("smoothed", torch.float64, smoothed), ("labels", torch.int32, labels),
                            ("sums", torch.float64, sums))}
    peaks = np.zeros((n, 21, 3))
    sd = None if sides is None else np.ascontiguousarray(sides, dtype=np.int32)
    torch.cuda.synchronize()
    _lib.check(_lib.lib().opb_hand_debug_post(G.ctx(), d.data_ptr(), n, 21, None if sd is None else sd.ctypes.data, h, w,
                                              mode, flags, *(None if v is None else v.data_ptr() for v in out.values()),
                                              peaks.ctypes.data))
    res = [peaks] + [v.cpu().numpy() for v in out.values() if v is not None]
    return res[0] if len(res) == 1 else res


def oracle(maps, mode):
    """maps (21, h, w) -> (21, 3): src/hand.py:59-75 (mode 0) or Batch_model.py:388-405 (mode 1)."""
    hwc = np.asarray(maps).transpose(1, 2, 0)
    return O.hand_postprocess(hwc.astype(np.float64)) if mode == 0 else O.batch_hand_postprocess(hwc.astype(np.float32))


def root_labels(binary):
    """scipy's 8-connected labels with every component named by its smallest raster index, -1 off the mask."""
    lab, n = ndi.label(binary, structure=EIGHT)
    flat = lab.ravel()
    first = np.full(n + 1, -1)
    idx = np.flatnonzero(flat)[::-1]
    first[flat[idx]] = idx                           # the last write per label is its smallest index
    return first[lab]


# ---- smoothing ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw", [(s, s) for s in range(1, 14)] + [(31, 31), (61, 95), (184, 184)])
def test_smoothing_bit_exact_at_every_side(hw):
    """Sides below the Gaussian radius (12) reflect more than once."""
    h, w = hw
    rng = np.random.default_rng(h * 1000 + w)
    maps = (rng.standard_normal((1, 21, h, w)) * 0.05).astype(np.float32)
    peaks, sm = post(maps, smoothed=True)
    for p in range(21):
        assert np.array_equal(sm[0, p], O.gaussian_sigma3(maps[0, p].astype(np.float64))), p
    assert np.array_equal(peaks[0], oracle(maps[0], 0))


# ---- labels -------------------------------------------------------------------------------------------------------------
def spiral(h, w):
    m = np.zeros((h, w), bool)
    y0, x0, y1, x1 = 0, 0, h - 1, w - 1
    while y0 <= y1 and x0 <= x1:
        m[y0, x0:x1 + 1] = m[y0:y1 + 1, x1] = m[y1, x0:x1 + 1] = True
        m[y0 + 2:y1 + 1, x0] = True
        y0, x0, y1, x1 = y0 + 2, x0 + 2, y1 - 2, x1 - 2
        if y0 <= y1 and x0 <= x1:
            m[y0, x0 - 2:x0] = True
            m[y0 - 1, x0 - 2] = True
    return m


def comb(h, w, tooth=3, vertical=True):
    m = np.zeros((h, w), bool)
    if vertical:
        m[h - 1, :] = True
        m[:, ::tooth] = True
    else:
        m[:, w - 1] = True
        m[::tooth, :] = True
    return m


def staircase(h, w, step=1):
    m = np.zeros((h, w), bool)
    for y in range(h):
        m[y, (y * step) % w] = True
    return m


def late_u(h, w):
    """Two long one-pixel arms that only meet in the last row (one component whose roots merge at the very end),
    next to a second U lying sideways."""
    m = np.zeros((h, w), bool)
    m[:, 1] = m[:, w - 2] = True
    m[h - 1, 1:w - 1] = True
    return m


def label_shapes():
    rng = np.random.default_rng(7)
    shapes = {
        "spiral_129": spiral(129, 129), "spiral_40x300": spiral(40, 300),
        "comb_v": comb(70, 260), "comb_h": comb(260, 70, vertical=False), "comb_wide": comb(33, 257, tooth=2),
        "checker": (np.add.outer(np.arange(64), np.arange(200)) % 2 == 0),
        "checker_sparse": (np.add.outer(np.arange(48), np.arange(160)) % 4 == 0)
        & (np.arange(48)[:, None] % 2 == 0),
        "stairs": staircase(200, 129), "stairs2": staircase(90, 300, 3), "u": late_u(161, 257),
        "full": np.ones((97, 150), bool), "row": np.ones((1, 333), bool), "col": np.ones((333, 1), bool),
        "row_gaps": rng.random((1, 700)) < 0.7, "col_gaps": rng.random((700, 1)) < 0.7,
        "noise": rng.random((150, 290)) < 0.55,
    }
    return shapes


def test_label_shapes_reach_their_cases():
    s = label_shapes()
    n = {k: ndi.label(v, structure=EIGHT)[1] for k, v in s.items()}
    assert n["spiral_129"] == 1 and n["comb_v"] == 1 and n["comb_h"] == 1 and n["u"] == 1 and n["full"] == 1
    assert n["checker"] == 1 and ndi.label(s["checker"])[1] == s["checker"].sum()     # connected only diagonally
    assert n["stairs"] == 2 and n["stairs2"] > 2
    assert n["row_gaps"] > 50 and n["col_gaps"] > 50 and n["noise"] > 1
    # runs crossing the 32-lane, 128-column and 16-row seams of the launches
    assert s["spiral_129"][0, 31:33].all() and s["comb_v"][69, 127:129].all() and s["comb_h"][15:17, 69].all()


@pytest.mark.parametrize("name", sorted(label_shapes()))
def test_labels_equal_scipy(name):
    """Batch_hand thresholds the map as given, so a crafted mask reaches the labelling unchanged; every plane of the
    crop holds the shape, the ones after the first shifted by their index (wrapping)."""
    b = label_shapes()[name]
    rng = np.random.default_rng(len(name))
    maps = np.zeros((1, 21) + b.shape, np.float32)
    for p in range(21):
        bp = np.roll(b, p, axis=1 if b.shape[1] > 1 else 0)
        maps[0, p] = np.where(bp, 0.05 + 0.9 * rng.random(b.shape), 0.01).astype(np.float32)
    peaks, labels = post(maps, mode=1, labels=True)
    for p in range(21):
        assert np.array_equal(labels[0, p], root_labels(maps[0, p] > np.float32(0.035))), p
    assert np.array_equal(peaks[0], oracle(maps[0], 1))


# ---- near ties ----------------------------------------------------------------------------------------------------------
def blob(rng, bh, bw, lo=-12):
    """float32 values spanning 10^lo … 1 inside a one-pixel frame of 1.0 (keeps the smoothed mask covering the blob)."""
    v = (rng.random((bh, bw)) * 10.0 ** rng.uniform(lo, 0, (bh, bw))).astype(np.float32)
    v[0, :] = v[-1, :] = v[:, 0] = v[:, -1] = 1.0
    return v


def hand_copies(seed, H_=150, W_=200, n_planes=21):
    """Two translated copies of one blob per plane, >= 40 px apart and 20 px from the border, so that their smoothed
    neighbourhoods and hence components are identical."""
    rng = np.random.default_rng(seed)
    maps = np.zeros((1, 21, H_, W_), np.float32)
    for p in range(n_planes):
        bh, bw = rng.integers(6, 14, 2)
        b = blob(rng, bh, bw)
        for (y, x) in ((20 + rng.integers(0, 10), 20 + rng.integers(0, 30)),
                       (H_ - 20 - bh - rng.integers(0, 10), W_ - 20 - bw - rng.integers(0, 30))):
            maps[0, p, y:y + bh, x:x + bw] = b
    return maps


def two_component_sums(m, mode):
    binary = (O.gaussian_sigma3(m.astype(np.float64)) > O.HAND_THRE) if mode == 0 else m > np.float32(0.035)
    lab, n, sums = H.component_sums(m, binary, np.float64 if mode == 0 else np.float32)
    return lab, n, sums


def test_hand_translated_copies():
    """numpy's sums of the two copies tie (the reference takes the first copy), while float64 sums of the same values
    in other orders differ -- the order of the device's atomics decides nothing."""
    maps = hand_copies(11)
    reorder = 0
    for p in range(21):
        lab, n, sums = two_component_sums(maps[0, p], 0)
        assert n == 2 and sums[0] == sums[1]
        v = maps[0, p].astype(np.float64)[lab == 2]
        rng = np.random.default_rng(p)
        reorder += any(np.cumsum(rng.permutation(v))[-1] != sums[0] for _ in range(8))
    assert reorder >= 15
    ref = oracle(maps[0], 0)
    for _ in range(3):
        assert np.array_equal(post(maps)[0], ref)


def test_hand_same_values_other_raster_order():
    """The second component holds the first one's values in another raster order: numpy's sums differ in the last
    bits only, well inside the certification bound, so the exact path decides."""
    rng = np.random.default_rng(12)
    maps = hand_copies(12)
    near = 0
    for p in range(21):
        m = maps[0, p]
        lab, n, _ = two_component_sums(m, 0)
        ys, xs = np.nonzero((lab == 2) & (m > 0))
        inner = (m[ys, xs] < 1.0)                     # keep the frame, permute the interior
        m[ys[inner], xs[inner]] = rng.permutation(m[ys[inner], xs[inner]])
        lab, n, sums = two_component_sums(m, 0)
        assert n == 2
        vals = m.astype(np.float64)[lab > 0]
        B = H.bound(np.abs(vals).sum(), vals.size)
        assert abs(sums[0] - sums[1]) <= 2 * B
        near += sums[0] != sums[1]
    assert near >= 5
    ref = oracle(maps[0], 0)
    for _ in range(3):
        assert np.array_equal(post(maps)[0], ref)


def batch_pairs(seed, reversed_order):
    """Batch_hand: per plane components A (first in raster order) and B.  reversed_order = False: B is A with one
    value raised by one float32 ulp (float32 sums tie, the exact sums say B).  True: B holds A's values in another
    order, one of them raised by one ulp, chosen so that the float32 sums order A, B the other way round from the exact
    sums."""
    rng = np.random.default_rng(seed)
    maps = np.full((1, 21, 120, 180), 0.01, np.float32)
    for p in range(21):
        bh, bw = rng.integers(10, 40, 2)
        for _ in range(1000):
            a = (0.05 + 0.9 * rng.random((bh, bw))).astype(np.float32)
            b = rng.permutation(a.ravel()).reshape(a.shape) if reversed_order else a.copy()
            i, j = rng.integers(0, bh), rng.integers(0, bw)
            b[i, j] = np.nextafter(b[i, j], np.float32(2))
            s32 = (np.sum(a), np.sum(b))
            e = (a.astype(np.float64).sum(), b.astype(np.float64).sum())
            ok = (s32[0] == s32[1] and e[1] > e[0]) if not reversed_order else \
                (s32[0] != s32[1] and (s32[0] > s32[1]) != (e[0] > e[1]) and e[0] != e[1])
            if ok:
                break
        else:
            raise AssertionError("no pair found")
        maps[0, p, 5:5 + bh, 5:5 + bw] = a
        maps[0, p, 70:70 + bh, 100:100 + bw] = b
    return maps


@pytest.mark.parametrize("reversed_order", [False, True])
def test_batch_hand_near_ties(reversed_order):
    maps = batch_pairs(21 + reversed_order, reversed_order)
    for p in range(21):
        lab, n, sums = two_component_sums(maps[0, p], 1)
        exact = [maps[0, p].astype(np.float64)[lab == i].sum() for i in (1, 2)]
        assert n == 2 and exact[0] != exact[1]
        assert (sums[0] == sums[1]) if not reversed_order else ((sums[0] > sums[1]) != (exact[0] > exact[1]))
    ref = oracle(maps[0], 1)
    for _ in range(3):
        assert np.array_equal(post(maps, mode=1)[0], ref)


def many_copies(n_copies=200, side=736):
    """n_copies identical blobs (values 1e-12 … 1) on a grid of a side x side map: every component ties, so every
    one of them is a contender."""
    rng = np.random.default_rng(31)
    maps = np.zeros((1, 21, side, side), np.float32)
    b = blob(rng, 8, 8)
    cols = 15
    cell = (side - 40) // cols
    for k in range(n_copies):
        y, x = 20 + (k // cols) * cell, 20 + (k % cols) * cell
        maps[0, 0, y:y + 8, x:x + 8] = b
    maps[0, 1] = maps[0, 0, :, ::-1]
    return maps


def test_hand_many_identical_copies():
    maps = many_copies()
    lab, n, sums = two_component_sums(maps[0, 0], 0)
    assert n == 200 and len(set(sums)) == 1
    ref = oracle(maps[0], 0)
    assert ref[0, 2] == 1.0 and tuple(ref[0, :2]) == (20, 20)
    for _ in range(2):
        assert np.array_equal(post(maps)[0], ref)


# ---- forced exact mode --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1])
def test_forced_mode_sums_are_numpys(mode):
    maps = smooth_noise_maps(120, 150, 21, 1.0, 0.06, 41).transpose(2, 0, 1)[None].astype(np.float32)
    if mode == 1:
        maps = np.ascontiguousarray(O.blur5_fixed_order(maps[0].transpose(1, 2, 0)).transpose(2, 0, 1))[None]
    fast = post(maps, mode=mode)
    peaks, labels, sums = post(maps, mode=mode, flags=1, labels=True, sums=True)
    assert np.array_equal(peaks, fast) and np.array_equal(peaks[0], oracle(maps[0], mode))
    comps = 0
    for p in range(21):
        lab, n, ref = two_component_sums(maps[0, p], mode)
        roots = root_labels(lab > 0)
        assert np.array_equal(labels[0, p], roots)
        for i in range(1, n + 1):
            r = int(roots[lab == i][0])
            got = sums[0, p].ravel()[r]
            assert (got if mode == 0 else np.float32(got)).tobytes() == ref[i - 1].tobytes()
        comps += n
    assert comps >= 100


# ---- ragged geometry ----------------------------------------------------------------------------------------------------
def test_sides_list_equals_single_crops_and_oracle():
    sides = [1, 7, 13, 64, 97, 150, 0, 736]
    wmax = max(sides)
    packed = np.zeros((len(sides), 21, wmax * wmax), np.float32)
    per = []
    for c, s in enumerate(sides):
        if s == 0:
            per.append(None)
            continue
        m = smooth_noise_maps(s, s, 21, 3 if s > 12 else 1, 0.05, 50 + c).transpose(2, 0, 1).astype(np.float32)
        if s == 736:
            m[5] = many_copies(40)[0, 0]              # near ties in the largest slot
        per.append(m)
        packed[c, :, :s * s] = m.reshape(21, -1)
    got = post(packed, sides=sides)
    hit = 0
    for c, m in enumerate(per):
        if m is None:
            assert not got[c].any()
            continue
        ref = oracle(m, 0)
        assert np.array_equal(got[c], post(m[None])[0]) and np.array_equal(got[c], ref), sides[c]
        hit += (ref[:, 2] != 0).sum()
    assert hit >= 60


# ---- edge values --------------------------------------------------------------------------------------------------------
def test_threshold_hit_exactly_and_empty():
    rng = np.random.default_rng(40)
    m = np.where(rng.random((1, 21, 50, 70)) < 0.5, np.float32(0.035), np.float32(0.2)).astype(np.float32)
    m[0, 3] = 0.035                                  # the whole plane sits on the threshold: nothing is kept
    m[0, 4] = 0.0
    ref = oracle(m[0], 1)
    assert not ref[3].any() and not ref[4].any() and ref[0, 2] == np.float32(0.2)
    assert np.array_equal(post(m, mode=1)[0], ref)
    assert not post(np.zeros((2, 21, 30, 30), np.float32)).any()
    # Hand: a constant plane whose smoothing lands on either side of 0.03
    c = np.zeros((1, 21, 40, 40), np.float32)
    for p in range(21):
        c[0, p] = np.float32(0.03) + np.float32(p - 10) * np.float32(1e-9)
    assert np.array_equal(post(c)[0], oracle(c[0], 0))


def nonpositive_component_maps():
    """A positive spike next to a deeper negative one (a horizontal dipole) near the top-left corner: the smoothing is
    above the threshold a few pixels to the left, and below it at the spike itself.  The component's raw values are
    then set slightly negative (which leaves the mask as it is), so the winning component holds no positive value and
    the reference takes the first pixel, in raster order, whose kept value is 0: the first one of row 0 past it."""
    maps = np.zeros((1, 21, 60, 60), np.float32)
    spots = ((0, 4), (1, 5), (2, 6), (0, 6), (3, 7))
    for p in range(21):
        y, x = spots[p % len(spots)]
        m = maps[0, p]
        m[y, x] = 60.0
        m[y, x + 1] = -78.0
        comp = O.gaussian_sigma3(m.astype(np.float64)) > O.HAND_THRE
        m[comp] = np.float32(-1e-4 * (1 + p // len(spots)))
    return maps


def test_component_of_nonpositive_values():
    maps = nonpositive_component_maps()
    ref = oracle(maps[0], 0)
    reached = 0
    for p in range(21):
        m = maps[0, p].astype(np.float64)
        lab, n, sums = two_component_sums(maps[0, p], 0)
        best = int(np.argmax(sums)) + 1
        if n >= 1 and (m[lab == best] <= 0).all() and (ref[p, 0], ref[p, 1]) != (0, 0):
            reached += 1
    assert reached >= 10
    assert np.array_equal(post(maps)[0], ref)
