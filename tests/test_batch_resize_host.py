"""CPU checks of the tap tables Batch_body / Batch_hand resize with, against the installed torch's own
F.interpolate(mode="bicubic") weights (tests/batch_resize_ref.py):
  - the front-end tables (F.interpolate(scale_factor=184 / H)) and the map side's x8 and size-mode tables equal torch's
    weights bit for bit, the composite map tables are the float64 operator rounded once;
  - a float32 stand-in of the device's front-end chain on those tables passes the per-element bound of
    batch_resize_ref, on float and uint8 frames;
  - the bound rejects the stand-in with each of the ways the front end could be subtly wrong: OpenCV's taps, the step
    in / out instead of 1 / scale_factor, align_corners=True, A = -0.5, zero padding instead of clamped taps, a missing
    -0.5, a missing / 255, swapped B / R channels; and the map side with OpenCV's operator.
The weights pinned here are those of torch's CPU kernel.  torch's CUDA kernel, which the reference runs, rounds its
polynomials in another order: on a B200 its weights differ from these by at most 1.27e-7 (about one ulp of 1.0) on
every geometry below, a residual far inside the bound's per-element slack."""
import numpy as np
import pytest

from oracle import openpose_oracle as O
from pytorch_openpose_b200 import _lib
from tests import batch_resize_ref as BR
from tests import composite_ref as R

# frames: common sizes, heights whose resize has 183 rows (int(H * (184 / H)) == 183), an upscaling front, a narrow one
FRONTS = [(720, 1280), (1080, 1920), (480, 640), (2160, 3840),
          (43, 77), (86, 128), (172, 300), (344, 640), (688, 1280), (715, 1280), (729, 1296),
          (97, 131), (200, 33)]


def lib_taps(src, dst, scale_factor):
    first = np.zeros(dst, np.int32)
    coef = np.zeros((dst, 4), np.float32)
    _lib.check(_lib.lib().opb_debug_batch_resize_taps(src, dst, float(scale_factor), first.ctypes.data, coef.ctypes.data))
    return first, coef


def lib_composite(n_net, n_resized, n_orig):
    first = np.zeros(n_orig, np.int32)
    w6 = np.zeros((n_orig, 6), np.float32)
    _lib.check(_lib.lib().opb_debug_batch_composite_taps(n_net, n_resized, n_orig, first.ctypes.data, w6.ctypes.data))
    return first, w6


def cv2_taps(src, dst, scale):
    first = np.zeros(dst, np.int32)
    coef = np.zeros((dst, 4), np.float32)
    _lib.check(_lib.lib().opb_debug_resize_taps(src, dst, float(scale), first.ctypes.data, coef.ctypes.data))
    return first, coef


def py_taps(src, dst, step, A=-0.75, align_corners=False):
    """torch's construction in plain float32 with knobs for the mutations (not bit-exact: fma-free)"""
    f32 = np.float32
    A = f32(A)
    d = np.arange(dst, dtype=np.float32)
    r = (f32(step) * d) if align_corners else (f32(step) * (d + f32(0.5)) - f32(0.5))
    i = np.minimum(np.floor(r).astype(np.int64), src - 1)
    t = np.clip(r - i.astype(np.float32), 0, 1).astype(np.float32)
    cc1 = lambda x: ((A + f32(2)) * x - (A + f32(3))) * x * x + f32(1)
    cc2 = lambda x: ((A * x - f32(5) * A) * x + f32(8) * A) * x - f32(4) * A
    coef = np.stack([cc2(t + f32(1)), cc1(t), cc1(f32(1) - t), cc2(f32(2) - t)], 1).astype(np.float32)
    return (i - 1).astype(np.int32), coef


def front_tables(H, W, which="lib"):
    """(x taps, y taps) of Batch_body's front end for an H x W frame"""
    scale, h, w, _, _ = O.batch_size_pad(O.BATCH_BODY_SCALE, H, W)
    if which == "lib":
        return lib_taps(W, w, scale), lib_taps(H, h, scale)
    if which == "cv2":
        return cv2_taps(W, w, 1.0 / scale), cv2_taps(H, h, 1.0 / scale)
    if which == "in_out":
        return py_taps(W, w, np.float32(W) / np.float32(w)), py_taps(H, h, np.float32(H) / np.float32(h))
    if which == "align_corners":
        return (py_taps(W, w, (W - 1) / (w - 1), align_corners=True),
                py_taps(H, h, (H - 1) / (h - 1), align_corners=True))
    if which == "A=-0.5":
        return py_taps(W, w, 1.0 / scale, A=-0.5), py_taps(H, h, 1.0 / scale, A=-0.5)
    raise ValueError(which)


def standin(frames, tx, ty, zero_pad=False, shift=True, div255=True, swap_rb=False):
    """The device chain (prepost.cu preprocess_f32_kernel, --fmad=false) in float32: x pass over the 4 column taps,
    y pass over the 4 row taps, each product and sum rounded, minus 0.5, bf16.  frames: (n, 3, H, W) float32 or
    (n, H, W, 3) uint8.  The keyword arguments are the mutations.  Returns (n, 3, h, w) float64 of bf16 values."""
    f = np.asarray(frames)
    if f.dtype == np.uint8:
        x = f.astype(np.float32)
        x = (x / np.float32(255)) if div255 else x
        x = x.transpose(0, 3, 1, 2)
    else:
        x = f.astype(np.float32)
    if swap_rb:
        x = x[:, ::-1]
    H, W = x.shape[2:]
    (xf, xc), (yf, yc) = tx, ty

    def taps(first, coef, n):
        idx = first[:, None] + np.arange(4)[None, :]
        c = coef.copy()
        if zero_pad:
            c[(idx < 0) | (idx > n - 1)] = 0
        return np.clip(idx, 0, n - 1), c

    xi, cx = taps(xf, xc, W)
    yi, cy = taps(yf, yc, H)
    t = x[..., xi[:, 0]] * cx[:, 0]
    for j in range(1, 4):
        t = t + x[..., xi[:, j]] * cx[:, j]                       # (n, 3, H, w)
    acc = np.zeros(x.shape[:2] + (len(yf), len(xf)), np.float32)
    for i in range(4):
        acc = acc + t[:, :, yi[:, i], :] * cy[:, i][:, None]
    r = (acc - np.float32(0.5)) if shift else acc
    return BR.bf16_rn(r)


def noise_frames(H, W, n=1, u8=False, seed=0):
    rng = np.random.default_rng(seed)
    if u8:
        return rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)
    return rng.random((n, 3, H, W), dtype=np.float32)


def front_ref(frames, H, W):
    h, w, wy, wx = BR.front_operators(H, W)
    return BR.front_reference(BR.frames_f32(frames), wy, wx)


def verdict(got, ref, mag):
    bad, amb = BR.front_check(got, ref, mag)
    return int(bad.sum()), float(amb.mean())


# ---- tables ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,W", FRONTS)
def test_front_tables_equal_torch(H, W):
    scale, h, w, _, _ = O.batch_size_pad(O.BATCH_BODY_SCALE, H, W)
    if H in (43, 86, 172, 344, 688, 715, 729):
        assert h == 183
    (xf, xc), (yf, yc) = front_tables(H, W)
    for first, coef, n, m in ((xf, xc, W, w), (yf, yc, H, h)):
        ref = BR.torch_matrix(n, scale_factor=scale)
        assert ref.shape == (m, n)
        got = BR.dense(first, coef, n)
        assert np.array_equal(got, ref), "%dx%d: %d weights differ, max %.3g" % (
            H, W, int((got != ref).sum()), np.abs(got - ref).max())


@pytest.mark.parametrize("H,W", FRONTS)
def test_map_tables_equal_torch(H, W):
    _, h, w, _, _ = O.batch_size_pad(O.BATCH_BODY_SCALE, H, W)
    for n_res, n_orig in ((w, W), (h, H)):
        n_net = -(-n_res // 8)
        assert np.array_equal(BR.dense(*lib_taps(n_net, 8 * n_net, 8.0), n_net), BR.torch_matrix(n_net, scale_factor=8.0))
        assert np.array_equal(BR.dense(*lib_taps(n_res, n_orig, 0.0), n_res), BR.torch_matrix(n_res, n_out=n_orig))
        # the composite tables: the exact composite rounded once, within 2 u |S| |X8| of the reference operator S X8
        # (batch_resize_ref's docstring)
        S, X8 = BR.torch_matrix(n_res, n_out=n_orig), BR.x8_then_crop(n_net, n_res)
        A, Aabs = S @ X8, np.abs(S) @ np.abs(X8)
        first, w6 = lib_composite(n_net, n_res, n_orig)
        got = np.zeros_like(A)
        rows = np.arange(n_orig)
        for k in range(6):
            got[rows, np.minimum(first + k, n_net - 1)] += w6[:, k]
        assert np.all(np.abs(got - A) <= 1.0001 * R.U * (np.abs(A) + 2 * Aabs))


def test_hand_maps_are_the_x8_upsample():
    """Batch_hand: the crop is not resized; the map side's size-mode resize is the identity"""
    for side in (64, 184, 368):
        assert np.array_equal(BR.map_operator(side // 8, side, side), BR.torch_matrix(side // 8, scale_factor=8.0))


# ---- front-end chain against the bound -----------------------------------------------------------------------------------
@pytest.mark.parametrize("H,W", [(720, 1280), (1080, 1920), (715, 1280), (97, 131), (200, 33)])
@pytest.mark.parametrize("u8", [False, True])
def test_standin_within_bound(H, W, u8):
    frames = noise_frames(H, W, u8=u8, seed=H + W)
    ref, mag = front_ref(frames, H, W)
    got = standin(frames, *front_tables(H, W))
    nbad, amb = verdict(got, ref, mag)
    assert nbad == 0 and amb < 0.01, (nbad, amb)


@pytest.mark.parametrize("H,W", [(720, 1280), (1080, 1920)])
def test_bound_rejects_opencv_tables(H, W):
    frames = noise_frames(H, W, seed=1)
    ref, mag = front_ref(frames, H, W)
    nbad, _ = verdict(standin(frames, *front_tables(H, W, "cv2")), ref, mag)
    assert nbad > 0


@pytest.mark.parametrize("which", ["in_out", "align_corners", "A=-0.5"])
def test_bound_rejects_wrong_taps(which):
    H, W = 720, 1280
    frames = noise_frames(H, W, seed=2)
    ref, mag = front_ref(frames, H, W)
    nbad, _ = verdict(standin(frames, *front_tables(H, W, which)), ref, mag)
    assert nbad > 0


def test_bound_rejects_zero_padding():
    """upscaling (97 x 131 -> 184 x 248): the first and last outputs have taps outside the frame"""
    H, W = 97, 131
    frames = np.zeros((1, 3, H, W), np.float32)
    frames[:, :, 0, :] = frames[:, :, -1, :] = frames[:, :, :, 0] = frames[:, :, :, -1] = 1.0
    ref, mag = front_ref(frames, H, W)
    assert verdict(standin(frames, *front_tables(H, W)), ref, mag)[0] == 0
    assert verdict(standin(frames, *front_tables(H, W), zero_pad=True), ref, mag)[0] > 0


@pytest.mark.parametrize("mutation", ["shift", "div255", "swap_rb"])
def test_bound_rejects_chain_mutations(mutation):
    H, W = 480, 640
    frames = noise_frames(H, W, u8=True, seed=3)
    ref, mag = front_ref(frames, H, W)
    kw = {"shift": dict(shift=False), "div255": dict(div255=False), "swap_rb": dict(swap_rb=True)}[mutation]
    assert verdict(standin(frames, *front_tables(H, W), **kw), ref, mag)[0] > 0


# ---- map side ----------------------------------------------------------------------------------------------------------
def map_dims(H, W):
    _, h, w, _, _ = O.batch_size_pad(O.BATCH_BODY_SCALE, H, W)
    return [(h, w, -(-h // 8), -(-w // 8))]


@pytest.mark.parametrize("H,W", [(720, 1280), (97, 131), (200, 33)])
def test_map_standin_within_torch_bound(H, W):
    dims = map_dims(H, W)
    ops = BR.map_operators(H, W, dims)
    rng = np.random.default_rng(H)
    nets = [rng.standard_normal((ho, wo, 4)).astype(np.float32) for _, _, ho, wo in dims]
    assert R.excess(R.standin(nets, ops), nets, ops, BR.MAP_EXTRA_ROUNDINGS) <= 1.0


def test_map_bound_rejects_opencv_operator():
    H, W = 720, 1280
    dims = map_dims(H, W)
    rng = np.random.default_rng(4)
    nets = [rng.standard_normal((ho, wo, 4)).astype(np.float32) for _, _, ho, wo in dims]
    assert R.excess(R.standin(nets, R.axis_operators(H, W, dims)), nets, BR.map_operators(H, W, dims),
                    BR.MAP_EXTRA_ROUNDINGS) > 1.0
