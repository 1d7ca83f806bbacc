"""The post-processing Body and Batch_body run in production -- tile bounds, the fused peak kernel that evaluates the
averaged heat map from the stride-8 net outputs (composite source), the PAF sampled through composite_at2 -- on crafted
net outputs, through the frame plan a real call of that geometry builds (opb_body_debug_post_submit skips only the
upload, the front end and the CNN).

Per frame:
  - the planes of opb_body_maps are within the float64 bound of tests/composite_ref.py, with OpenCV's operator for Body
    and torch's (tests/batch_resize_ref.py) for Batch_body;
  - Body: candidates and part_begin equal O.find_peaks on those planes bit for bit, each candidate's score is the plane
    value at its (y, x) (the composite values equal the materialised ones), subsets equal O.match_limbs + O.assemble;
  - Batch_body: opb_batch_maps equals O.blur5_fixed_order of the heat planes, results equal O.batch_body_postprocess.
Every content family asserts, on oracle-side quantities, that it reaches the case it is written for."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import openpose_oracle as O
from pytorch_openpose_b200 import _lib
from tests import batch_resize_ref as BR
from tests import composite_ref as R

pytestmark = pytest.mark.gpu

THRE1, THRE2 = 0.1, 0.05


@pytest.fixture(scope="module")
def sess():
    net = _lib.Net(_lib.NET_BODY, O.make_weights("body", 0))
    return net.session()


def geometry(H, W, scales, mode):
    """per-scale (h, w, ho, wo) of the plan and whether its heat maps go through the fused (composite) peak kernel"""
    sc, ns = _lib.scales_array(scales)
    hw = (ctypes.c_int * (2 * ns))()
    fused = ctypes.c_int()
    _lib.check(_lib.lib().opb_body_debug_post_dims(H, W, sc, ns, mode, hw, ctypes.byref(fused)))
    if mode == 0:
        hws = [(p["h"], p["w"]) for p in O.scale_plan(H, W, scales)]
    else:
        _, h, w, _, _ = O.batch_size_pad(scales[0], H, W)
        hws = [(h, w)]
    dims = [(h, w, hw[2 * i], hw[2 * i + 1]) for i, (h, w) in enumerate(hws)]
    for h, w, ho, wo in dims:
        assert (ho, wo) == (-(-h // 8), -(-w // 8))
    return dims, fused.value


def run(sess, H, W, scales, mode, heat, paf):
    """heat / paf: per scale (n, ho, wo, 19 / 38) net outputs.  -> per-frame results, heat / PAF planes, blurred planes"""
    L = _lib.lib()
    n = heat[0].shape[0]
    hp, pp = [], []
    for h, p in zip(heat, paf):
        a = np.zeros(h.shape[:3] + (24,), np.float32)
        a[..., :19] = h
        b = np.zeros(p.shape[:3] + (40,), np.float32)
        b[..., :38] = p
        hp.append(a)
        pp.append(b)
    sc, ns = _lib.scales_array(scales)
    hptr = (ctypes.c_void_p * ns)(*[a.ctypes.data for a in hp])
    pptr = (ctypes.c_void_p * ns)(*[b.ctypes.data for b in pp])
    torch.cuda.synchronize()
    _lib.check(L.opb_body_debug_post_submit(sess.handle, n, H, W, sc, ns, mode, hptr, pptr))
    nc, nsub, st = (ctypes.c_int * n)(), (ctypes.c_int * n)(), (ctypes.c_int * n)()
    rc = L.opb_body_wait_batch(sess.handle, nc, nsub, st)
    if rc != _lib.OPB_ERR_SUBSET_INDEX:
        _lib.check(rc)
    frames = []
    for f in range(n):
        cand, sub = np.zeros((max(nc[f], 1), 4)), np.zeros((max(nsub[f], 1), 20))
        _lib.check(L.opb_body_fetch_frame(sess.handle, f, cand.ctypes.data, nc[f], sub.ctypes.data, nsub[f]))
        pb = (ctypes.c_int * 19)()
        _lib.check(L.opb_body_debug_part_begin(sess.handle, f, pb))
        frames.append(dict(cand=cand[:nc[f]], subset=sub[:nsub[f]], part_begin=list(pb), status=st[f]))
    hm, pm = np.zeros((n, 19, H, W), np.float32), np.zeros((n, 38, H, W), np.float32)
    _lib.check(L.opb_body_maps(sess.handle, hm.ctypes.data, pm.ctypes.data))
    bl = None
    if mode == 1:
        bl = np.zeros((n, 19, H, W), np.float32)
        _lib.check(L.opb_batch_maps(sess.handle, bl.ctypes.data))
    return frames, hm, pm, bl


def verify(sess, H, W, scales, mode, heat, paf, fused):
    """Runs one batch and checks it against the oracle.  Returns per frame the oracle-side quantities the coverage
    assertions use: peaks, the map NMS ran on (18, H, W), the PAF planes (H, W, 38) float64 and the reference subset."""
    dims, got_fused = geometry(H, W, scales, mode)
    assert got_fused == fused
    frames, hm, pm, bl = run(sess, H, W, scales, mode, heat, paf)
    # Body resizes like cv2, Batch_body like torch's F.interpolate (tests/batch_resize_ref.py)
    if mode == 0:
        ops, extra = R.axis_operators(H, W, dims), 0
    else:
        ops, extra = BR.map_operators(H, W, dims), BR.MAP_EXTRA_ROUNDINGS
    out = []
    for i, fr in enumerate(frames):
        R.assert_within_bound(hm[i], [h[i] for h in heat], ops, "heat, frame %d" % i, extra)
        R.assert_within_bound(pm[i], [p[i] for p in paf], ops, "paf, frame %d" % i, extra)
        heat64 = hm[i].transpose(1, 2, 0).astype(np.float64)
        paf64 = pm[i].transpose(1, 2, 0).astype(np.float64)
        if mode == 0:
            sms = []
            peaks = O.find_peaks(heat64, THRE1, smooth=lambda m: sms.append(O.gaussian_sigma3(m)) or sms[-1])
            nms, scored = np.stack(sms), hm[i]
        else:
            blurred = O.blur5_fixed_order(hm[i].transpose(1, 2, 0))
            assert np.array_equal(bl[i].transpose(1, 2, 0), blurred)
            peaks = O.batch_find_peaks(blurred, THRE1)
            nms = scored = blurred.transpose(2, 0, 1)
        lens = [len(p) for p in peaks]
        assert np.array_equal(fr["cand"], np.concatenate(peaks)), "frame %d: candidates differ" % i
        assert fr["part_begin"] == [int(v) for v in np.cumsum([0] + lens)]
        part = np.repeat(np.arange(18), lens)
        xs, ys = fr["cand"][:, 0].astype(int), fr["cand"][:, 1].astype(int)
        assert np.array_equal(fr["cand"][:, 2], scored[part, ys, xs].astype(np.float64))
        subset_ref = None
        try:
            if mode == 0:
                conns, special = O.match_limbs(peaks, paf64, H, THRE2)
                _, subset_ref = O.assemble(peaks, conns, special)
            else:
                _, subset_ref = O.batch_body_postprocess(blurred, pm[i].transpose(1, 2, 0), THRE1, THRE2)
        except IndexError:
            assert fr["status"] == _lib.OPB_ERR_SUBSET_INDEX
        if subset_ref is not None:
            assert fr["status"] == _lib.OPB_OK
            assert np.array_equal(fr["subset"], subset_ref), "frame %d: subsets differ" % i
        out.append(dict(peaks=peaks, nms=nms, paf=paf64, subset=subset_ref))
    return out


# ---- content: drawn at each scale's net output size ------------------------------------------------------------------
def blank(dims, n):
    heat = [np.zeros((n, ho, wo, 19), np.float32) for _, _, ho, wo in dims]
    paf = [np.zeros((n, ho, wo, 38), np.float32) for _, _, ho, wo in dims]
    for h in heat:
        h[..., 18] = 1.0
    return heat, paf


def bump(heat, dims, H, W, f, ch, x, y, amp, sigma):
    """a Gaussian of full-resolution centre (x, y) and width sigma (px), sampled on every scale's net output grid"""
    for a, (h, w, ho, wo) in zip(heat, dims):
        kx, ky = w / (8.0 * W), h / (8.0 * H)                 # full-resolution px -> net output cells
        u, v = (x + 0.5) * kx - 0.5, (y + 0.5) * ky - 0.5
        jj, ii = np.arange(wo), np.arange(ho)
        g = np.exp(-0.5 * ((ii[:, None] - v) / (sigma * ky)) ** 2 - 0.5 * ((jj[None, :] - u) / (sigma * kx)) ** 2)
        a[f, :, :, ch] += (amp * g).astype(np.float32)


# 0.1 as float32 rounds up (0.1f = 0.1 + 1.5e-9); noise is centred on the midpoint between 0.1f and its lower
# neighbour so that even delta = 1e-9 straddles the threshold instead of rounding to 0.1f everywhere
NEAR = (np.float64(np.float32(0.1)) + np.float64(np.nextafter(np.float32(0.1), np.float32(0)))) / 2


# Batch_body thresholds the 5x5-blurred map, whose taps sum to 0.9967
NEAR_BLURRED = 0.1 / float(O.BLUR5.astype(np.float64).sum())


def fill_near(heat, paf, f, delta, seed, center=NEAR):
    """family 1: 0.1 + delta * noise on every part map"""
    rng = np.random.default_rng(seed)
    for h, p in zip(heat, paf):
        h[f, :, :, :18] = (center + delta * rng.standard_normal(h.shape[1:3] + (18,))).astype(np.float32)
        p[f] = (0.2 * rng.standard_normal(p.shape[1:])).astype(np.float32)


def fill_ties(heat, f):
    """family 2 (pure x8 geometry, one scale): constant blocks and mirror-symmetric pairs of exactly representable
    values -- plateaus and equal neighbours in the smoothed maps"""
    h = heat[0]
    for part in range(18):
        r, c = 4 + part % 3, 4 + part % 5
        h[f, r:r + 10, c:c + 12, part] = 0.5                                # constant block: a plateau of the smoothed map
        h[f, r + 20, c + 30:c + 32, part] = 0.25                            # two equal cells: a mirror-symmetric ridge
        h[f, r + 26, c + 40, part] = 0.125                                  # a lone cell
        h[f, r + 30:r + 32, c + 50:c + 52, part] = 0.375                    # 2x2 block
        h[f, r + 22:r + 30, c + 60:c + 68, part] = 0.1                      # a constant block at the threshold


def fill_high_range(heat, dims, H, W, f, x0, y0, seed):
    """family 3: in the tile window at (x0, y0) (64 x 32 px), one net output sample of 1e3..1e4 and bumps near the
    threshold 32..48 px away, on every part"""
    rng = np.random.default_rng(seed)
    for part in range(18):
        big = float(10 ** (3 + part / 17.0))
        for h, (hh, w, ho, wo) in zip(heat, dims):
            r = int(round((y0 + 8.5) * hh / (8.0 * H) - 0.5))
            c = int(round((x0 + 8.5) * w / (8.0 * W) - 0.5))
            h[f, r, c, part] = big
        for k in range(3):
            amp = 0.1 + 0.004 * (k - 1) + 1e-4 * rng.standard_normal()
            bump(heat, dims, H, W, f, part, x0 + 40 + 7 * k, y0 + 8 + 8 * k, amp / 0.55, 6.0)


def fill_seams(heat, dims, H, W, f, xt, yt):
    """family 4: bumps centred so that peaks land on the columns xt and the rows yt; each part is shifted by its own
    sub-pixel offset, so some part lands exactly on every target"""
    sigma = max([6.0] + [1.2 * 8 * max(W / w, H / h) for h, w, _, _ in dims])    # resolved by the coarsest grid
    for part in range(18):
        d = (part % 6 - 2.5) * 0.2
        for k, x in enumerate(xt):
            bump(heat, dims, H, W, f, part, x + d, (0.15 + 0.7 * k / (len(xt) - 1)) * H + d, 0.6, sigma)
        for k, y in enumerate(yt):
            bump(heat, dims, H, W, f, part, (0.15 + 0.22 * k) * W + d, y + d, 0.6, sigma)


def fill_level(heat, paf, f, level, seed):
    """family 5: smooth noise entirely below (level < thre1) or above the threshold"""
    rng = np.random.default_rng(seed)
    for h, p in zip(heat, paf):
        h[f, :, :, :18] = (level + 0.02 * rng.random(h.shape[1:3] + (18,))).astype(np.float32)
        p[f] = (0.1 * rng.standard_normal(p.shape[1:])).astype(np.float32)


def fill_persons(heat, paf, dims, H, W, f, grid, seed, pairs=5, row=0.95):
    """family 6: O.synthetic_scene drawn on the top three quarters of each scale's grid, and below it `pairs` isolated
    neck / right-shoulder pairs on the row `row` H; the PAF of limb 0 is the constant field (0.05, 0), so the
    projections sampled between the pairs sit at thre2 = 0.05 where the row's resampling weights carry 0.05f through
    unchanged (cv2's last tap is 1 minus the other three, torch's is a polynomial of its own, so that depends on the
    row)"""
    cx, cy = O.PAF_CH[0]
    for h, p, (hh, w, ho, wo) in zip(heat, paf, dims):
        top = max(4, (3 * ho) // 4)
        sh, sp, _ = O.synthetic_scene(top, wo, grid, seed=seed, jitter=0.0)
        h[f, :top] = sh.astype(np.float32)
        p[f, :top] = sp.astype(np.float32)
        p[f, :, :, cx] = np.float32(THRE2)                                # limb 0 everywhere: no edge of the field
        p[f, :, :, cy] = 0.0                                               # overshoots near the pairs
    for k in range(pairs):
        x = (0.05 + 0.19 * k) * W
        for part, dx in ((1, 0.0), (2, 0.12 * W)):
            bump(heat, dims, H, W, f, part, x + dx, round(row * H), 0.8, max(6.0, 0.012 * H))


def thre2_samples(peaks, paf, H):
    """number of PAF samples (score_pairs' projections) within 1e-9 of thre2, over all limbs and candidate pairs"""
    n = 0
    for k, (a, b) in enumerate(O.LIMB_SEQ):
        A, B = peaks[a - 1], peaks[b - 1]
        if len(A) == 0 or len(B) == 0:
            continue
        vx, vy = B[None, :, 0] - A[:, None, 0], B[None, :, 1] - A[:, None, 1]
        norm = np.sqrt(vx * vx + vy * vy) + 1e-10
        t = np.arange(O.MID_NUM)[None, None, :]
        px = t * (vx / (O.MID_NUM - 1))[..., None] + A[:, None, None, 0]
        py = t * (vy / (O.MID_NUM - 1))[..., None] + A[:, None, None, 1]
        px[..., -1] = B[None, :, 0]
        py[..., -1] = B[None, :, 1]
        xi, yi = np.rint(px).astype(int), np.rint(py).astype(int)
        cx, cy = O.PAF_CH[k]
        dots = paf[yi, xi, cx] * (vx / norm)[..., None] + paf[yi, xi, cy] * (vy / norm)[..., None]
        n += int((np.abs(dots - THRE2) < 1e-9).sum())
    return n


def near_maxima(nms, delta, thre=THRE1):
    """(accepted, rejected) 4-neighbour maxima (zero outside the map) with |value - thre| < 10 delta"""
    z = np.pad(nms, ((0, 0), (1, 1), (1, 1)))
    c = z[:, 1:-1, 1:-1]
    m = (c >= z[:, :-2, 1:-1]) & (c >= z[:, 2:, 1:-1]) & (c >= z[:, 1:-1, :-2]) & (c >= z[:, 1:-1, 2:])
    m &= np.abs(c - thre) < 10 * delta
    above = c > (np.float32(thre) if nms.dtype == np.float32 else thre)
    return int((m & above).sum()), int((m & ~above).sum())


def has_equal_neighbour(peaks, nms):
    H, W = nms.shape[1:]
    for part, arr in enumerate(peaks):
        for x, y in arr[:, :2].astype(int):
            for dy, dx in ((-1, 0), (1, 0), (0, -1), (0, 1)):
                if 0 <= y + dy < H and 0 <= x + dx < W and nms[part, y + dy, x + dx] == nms[part, y, x]:
                    return True
    return False


def on_lines(peaks, xt, yt):
    allp = np.concatenate(peaks)
    return all((allp[:, 0] == x).any() for x in xt) and all((allp[:, 1] == y).any() for y in yt)


def in_window(peaks, x0, y0):
    """a peak in the window (tile + halo) of the 64 x 32 tile at (x0, y0), other than that of the large sample"""
    h = 13
    for arr in peaks:
        for x, y in arr[:, :2]:
            if x0 - h <= x < x0 + 64 + h and y0 - h <= y < y0 + 32 + h and max(abs(x - x0 - 8), abs(y - y0 - 8)) > 8:
                return True
    return False


def assemble_cover(res, H, W, at_thre2=True):
    assert sum(len(r["subset"]) for r in res if r["subset"] is not None) >= 3
    if at_thre2:
        assert sum(thre2_samples(r["peaks"], r["paf"], H) for r in res) >= 10


# ---- Body (mode 0) ---------------------------------------------------------------------------------------------------
X8 = (368, 656, (1.0,))          # pure x8 composite: the resize to the frame is the identity


@pytest.mark.parametrize("delta", [1e-9, 1e-6, 1e-3])
def test_near_threshold_x8(sess, delta):
    H, W, sc = X8
    dims, _ = geometry(H, W, sc, 0)
    heat, paf = blank(dims, 1)
    fill_near(heat, paf, 0, delta, int(-np.log10(delta)))
    r = verify(sess, H, W, sc, 0, heat, paf, fused=1)[0]
    acc, rej = near_maxima(r["nms"], delta)
    assert acc >= 20 and rej >= 20, (acc, rej)


def test_ties_and_plateaus_x8(sess):
    H, W, sc = X8
    dims, _ = geometry(H, W, sc, 0)
    heat, paf = blank(dims, 1)
    fill_ties(heat, 0)
    r = verify(sess, H, W, sc, 0, heat, paf, fused=1)[0]
    assert has_equal_neighbour(r["peaks"], r["nms"])


def test_seams_and_high_range_x8(sess):
    H, W, sc = X8
    dims, _ = geometry(H, W, sc, 0)
    heat, paf = blank(dims, 2)
    xt, yt = (0, 63, 64, W - 1), (0, 31, 32, H - 1)
    fill_seams(heat, dims, H, W, 0, xt, yt)
    fill_high_range(heat, dims, H, W, 1, 128, 96, 5)
    r = verify(sess, H, W, sc, 0, heat, paf, fused=1)
    assert on_lines(r[0]["peaks"], xt, yt)
    assert in_window(r[1]["peaks"], 128, 96)


def test_bench_geometry_persons_and_high_range(sess):
    H, W, sc = 720, 1280, (0.5, 1.0, 1.5, 2.0)
    dims, _ = geometry(H, W, sc, 0)
    heat, paf = blank(dims, 2)
    fill_persons(heat, paf, dims, H, W, 0, (4, 1), 1)
    fill_high_range(heat, dims, H, W, 1, 640, 352, 6)
    r = verify(sess, H, W, sc, 0, heat, paf, fused=1)
    assemble_cover(r[:1], H, W)
    assert in_window(r[1]["peaks"], 640, 352)


@pytest.mark.parametrize("scales,fused", [((0.5,), 1), ((0.5, 1.5), 0)])
def test_odd_width(sess, scales, fused):
    """97 x 131 (W % 4 != 0: the planes come from the generic y kernel).  At (0.5, 1.5) the footprint of a tile is too
    large for the fused kernel and the heat maps are materialised first."""
    H, W = 97, 131
    dims, _ = geometry(H, W, scales, 0)
    heat, paf = blank(dims, 4)
    xt, yt = (0, 63, 64, W - 1), (0, 31, 32, H - 1)
    fill_seams(heat, dims, H, W, 0, xt, yt)
    fill_near(heat, paf, 1, 1e-6, 7)
    fill_level(heat, paf, 2, 0.03, 8)
    fill_level(heat, paf, 3, 0.5, 9)
    r = verify(sess, H, W, scales, 0, heat, paf, fused=fused)
    assert on_lines(r[0]["peaks"], xt, yt)
    acc, rej = near_maxima(r[1]["nms"], 1e-6)
    assert acc >= 20 and rej >= 20, (acc, rej)
    assert sum(map(len, r[2]["peaks"])) == 0
    assert all(len(p) > 0 for p in r[3]["peaks"])


def test_eight_scales(sess):
    H, W, sc = 240, 320, tuple(float(s) for s in np.linspace(0.25, 1.0, 8))
    dims, _ = geometry(H, W, sc, 0)
    heat, paf = blank(dims, 2)
    fill_persons(heat, paf, dims, H, W, 0, (3, 1), 2)
    fill_near(heat, paf, 1, 1e-3, 3)
    r = verify(sess, H, W, sc, 0, heat, paf, fused=1)
    # eight fmaf chains of rounding: the constant field comes out a few ulps off 0.05, the samples straddle thre2 only
    # at ~1e-8
    assemble_cover(r[:1], H, W, at_thre2=False)
    acc, rej = near_maxima(r[1]["nms"], 1e-3)
    assert acc >= 20 and rej >= 20, (acc, rej)


def test_batch_of_five_different_frames(sess):
    H, W, sc = 240, 320, (0.5, 1.0)
    dims, _ = geometry(H, W, sc, 0)
    heat, paf = blank(dims, 5)
    xt, yt = (0, 63, 64, 127, 128, W - 1), (0, 31, 32, H - 1)
    fill_near(heat, paf, 0, 1e-6, 11)
    fill_persons(heat, paf, dims, H, W, 1, (3, 1), 12)
    fill_seams(heat, dims, H, W, 2, xt, yt)
    fill_high_range(heat, dims, H, W, 3, 64, 64, 13)
    fill_level(heat, paf, 4, 0.5, 14)
    r = verify(sess, H, W, sc, 0, heat, paf, fused=1)
    acc, rej = near_maxima(r[0]["nms"], 1e-6)
    assert acc >= 20 and rej >= 20, (acc, rej)
    assemble_cover(r[1:2], H, W)
    assert on_lines(r[2]["peaks"], xt, yt)
    assert in_window(r[3]["peaks"], 64, 64)


# ---- Batch_body (mode 1) ---------------------------------------------------------------------------------------------
# The maps are bounded with torch's resize operator (F.interpolate, tests/batch_resize_ref.py), which the reference
# applies and the batched plans' tables follow; OpenCV's operator is Body's.
def test_batch_body_720p_torch_resize(sess):
    H, W, sc = 720, 1280, (O.BATCH_BODY_SCALE,)
    dims, _ = geometry(H, W, sc, 1)
    heat, paf = blank(dims, 4)
    # 31 px net output cells: the column seams and borders are reached; near a row seam or border the coarse grid puts
    # the maximum a few rows off, so the rows are left to the Body cases
    xt, yt = (0, 63, 64, W - 1), ()
    # 1e-3: at 1e-6 the float32 rounding of the interpolated maps leaves ulp-sized local maxima all over the 5x5-blurred
    # map (Body's sigma-3 smoothing in float64 averages them out), hundreds of thousands of candidates per frame
    fill_near(heat, paf, 0, 1e-3, 21, NEAR_BLURRED)
    fill_persons(heat, paf, dims, H, W, 1, (4, 1), 22, row=0.94)
    fill_seams(heat, dims, H, W, 2, xt, yt)
    fill_high_range(heat, dims, H, W, 3, 640, 352, 23)
    r = verify(sess, H, W, sc, 1, heat, paf, fused=1)
    acc, rej = near_maxima(r[0]["nms"], 1e-3)
    assert acc >= 20 and rej >= 20, (acc, rej)
    assemble_cover(r[1:2], H, W)
    assert on_lines(r[2]["peaks"], xt, yt)
    assert in_window(r[3]["peaks"], 640, 352)


@pytest.mark.parametrize("H,W", [(97, 131), (200, 33)])
def test_batch_body_small_torch_resize(sess, H, W):
    sc = (O.BATCH_BODY_SCALE,)
    dims, _ = geometry(H, W, sc, 1)
    heat, paf = blank(dims, 3)
    fill_near(heat, paf, 0, 1e-3, 31, NEAR_BLURRED)
    fill_level(heat, paf, 1, 0.03, 32)
    fill_level(heat, paf, 2, 0.5, 33)
    r = verify(sess, H, W, sc, 1, heat, paf, fused=1)
    assert sum(map(len, r[1]["peaks"])) == 0
    assert all(len(p) > 0 for p in r[2]["peaks"])
