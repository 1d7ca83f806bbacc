"""The torch bicubic resizes of Batch_body / Batch_hand on the device, against the float64 references of
tests/batch_resize_ref.py built from the installed torch's own weights.

Front end (opb_batch_debug_input: the bf16 net input of the last batch):
  - Batch_body on float frames (submit) and uint8 frames (submit_frames): every element is a bf16 rounding of a value
    within the bound of ref - 0.5, the padding is exactly zero, fewer than 1 % of the elements are ambiguous (the bound
    straddles a bf16 rounding boundary), constant frames give bf16(c - 0.5) exactly;
  - Batch_hand crops are not resized: the input is bf16(x - 0.5) exactly.
Each batch mixes contents where a wrong tap shows: uniform noise, 0/1 checkerboards of 4-pixel cells (ref - 0.5
often lands near 0, where bf16 resolves ~1e-5), single bright pixels on the first / last rows and columns (clamped
taps), constants.

Map side (opb_body_debug_post_submit mode 1, crafted net outputs): the planes of opb_body_maps are within the bound of
torch's operator and candidates / subsets equal O.batch_body_postprocess on them (tests/test_gpu_fused_post.verify)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import openpose_oracle as O
from pytorch_openpose_b200 import _lib
from pytorch_openpose_b200.batch_model import Batch_body, Batch_hand
from tests import batch_resize_ref as BR
from tests import test_gpu_fused_post as FP
from tests.test_batch_resize_host import FRONTS

pytestmark = pytest.mark.gpu

CONSTANTS = (0.25, 0.8, 1.0)


@pytest.fixture(scope="module")
def body():
    return Batch_body(O.make_weights("body", 0))


@pytest.fixture(scope="module")
def hand():
    return Batch_hand(O.make_weights("hand", 0))


def net_input(est, n, hp, wp):
    """(n, 3, hp, wp) float64 values of the bf16 net input of the estimator's last batch"""
    bits = np.zeros((n, hp, wp, 3), np.uint16)
    _lib.check(_lib.lib().opb_batch_debug_input(est._session.handle, bits.ctypes.data))
    return (bits.astype(np.uint32) << 16).view(np.float32).astype(np.float64).transpose(0, 3, 1, 2)


def body_wait(est, n):
    """finish the batch; crafted frames on random weights may end in the reference's IndexError, which is not at issue"""
    nc, ns, st = (ctypes.c_int * n)(), (ctypes.c_int * n)(), (ctypes.c_int * n)()
    rc = _lib.lib().opb_body_wait_batch(est._session.handle, nc, ns, st)
    if rc != _lib.OPB_ERR_SUBSET_INDEX:
        _lib.check(rc)


def mixed_frames(H, W, seed, u8):
    """(n, 3, H, W) float32 in [0, 1]: noise, checkerboard, bright edge pixels, constants; uint8 frames are drawn on
    the 0..255 grid and returned as (n, H, W, 3) uint8"""
    rng = np.random.default_rng(seed)
    noise = rng.random((3, H, W))
    yy, xx = np.mgrid[:H, :W]
    # 4-pixel cells: a 1-pixel board resizes to ~0.5 everywhere, where the bound straddles bf16 boundaries
    checker = np.broadcast_to((((yy // 4) + (xx // 4)) % 2).astype(np.float64), (3, H, W))
    edges = np.zeros((3, H, W))
    for c, (y, x) in enumerate(((0, W // 3), (H - 1, (2 * W) // 3), (H // 2, 0))):
        edges[c, y, x] = 1.0
    edges[:, H // 3, W - 1] = 1.0
    edges[:, 0, 0] = edges[:, H - 1, W - 1] = 1.0
    frames = np.stack([noise, checker, edges] + [np.full((3, H, W), c) for c in CONSTANTS])
    if u8:
        return np.ascontiguousarray(np.rint(frames * 255).astype(np.uint8).transpose(0, 2, 3, 1))
    return frames.astype(np.float32)


def check_front(got, frames, H, W):
    """-> (bad elements, ambiguous fraction) of the resized part; asserts the padding and the constant frames"""
    h, w, wy, wx = BR.front_operators(H, W)
    ref, mag = BR.front_reference(BR.frames_f32(frames), wy, wx)
    body_part = got[:, :, :h, :w]
    assert np.all(got[:, :, h:, :] == 0) and np.all(got[:, :, :, w:] == 0), "padding is not zero"
    assert not np.signbit(got[:, :, h:, :]).any() and not np.signbit(got[:, :, :, w:]).any()
    bad, amb = BR.front_check(body_part, ref, mag)
    for k, c in enumerate(CONSTANTS):
        x = BR.frames_f32(frames)[3 + k, 0, 0, 0]
        assert np.all(body_part[3 + k] == BR.bf16_rn(np.float32(x) - np.float32(0.5))), "constant %g" % x
    return int(bad.sum()), float(amb.mean()), [int(b.sum()) for b in bad]


@pytest.mark.parametrize("H,W", FRONTS)
@pytest.mark.parametrize("u8", [False, True])
def test_batch_body_front_end(body, H, W, u8):
    frames = mixed_frames(H, W, H * W, u8)
    n = len(frames)
    _, h, w, pad_h, pad_w = O.batch_size_pad(O.BATCH_BODY_SCALE, H, W)
    torch.cuda.synchronize()
    if u8:
        body.submit_frames(frames)
    else:
        body.submit(frames)
    body_wait(body, n)
    got = net_input(body, n, h + pad_h, w + pad_w)
    nbad, amb, per_frame = check_front(got, frames, H, W)
    assert nbad == 0, "%dx%d: %d elements outside the bound (per frame %s)" % (H, W, nbad, per_frame)
    assert amb < 0.01, amb


@pytest.mark.parametrize("S", [64, 184, 368])
@pytest.mark.parametrize("u8", [False, True])
def test_batch_hand_front_end_is_exact(hand, S, u8):
    frames = mixed_frames(S, S, S, u8)
    n = len(frames)
    torch.cuda.synchronize()
    if u8:
        hand.submit_frames(frames)
    else:
        hand.submit(frames)
    hand.collect()
    got = net_input(hand, n, S, S)
    x = BR.frames_f32(frames)
    want = BR.bf16_rn((torch.from_numpy(x) - 0.5).numpy())
    assert np.array_equal(got, want)


# ---- map side -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sess():
    return _lib.Net(_lib.NET_BODY, O.make_weights("body", 0)).session()


def fill_noise(heat, paf, f, seed):
    """noise below the threshold on every map: bounds the planes everywhere, no candidates"""
    rng = np.random.default_rng(seed)
    for h, p in zip(heat, paf):
        h[f, :, :, :18] = (0.08 * rng.random(h.shape[1:3] + (18,))).astype(np.float32)
        p[f] = rng.standard_normal(p.shape[1:]).astype(np.float32)


def fill_edge_impulses(heat, paf, f):
    """single net samples on the first / last net rows and columns (the clamped taps of both passes)"""
    for h, p in zip(heat, paf):
        ho, wo = h.shape[1:3]
        for part, (r, c) in enumerate(((0, wo // 2), (ho - 1, wo // 3), (ho // 2, 0), (ho // 3, wo - 1),
                                      (0, 0), (ho - 1, wo - 1))):
            h[f, r, c, part] = 1.0
            p[f, r, c, 2 * part] = 1.0


@pytest.mark.parametrize("H,W", [(720, 1280), (1080, 1920), (715, 1280), (97, 131), (200, 33)])
def test_batch_body_maps(sess, H, W):
    sc = (O.BATCH_BODY_SCALE,)
    dims, fused = FP.geometry(H, W, sc, 1)
    heat, paf = FP.blank(dims, 3)
    fill_noise(heat, paf, 0, H)
    fill_edge_impulses(heat, paf, 1)
    FP.fill_high_range(heat, dims, H, W, 2, min(64, W // 2), min(32, H // 2), W)
    FP.verify(sess, H, W, sc, 1, heat, paf, fused)
