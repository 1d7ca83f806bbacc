"""float64 references and error bounds for the torch bicubic resizes of Batch_body / Batch_hand
(srcmx/Batch_model.py:153-155, :173-176, :377): F.interpolate(mode="bicubic", align_corners=False) on float32 tensors.

Weights.  torch_matrix takes torch's float32 weights from the installed torch itself: the impulse responses of
F.interpolate on the identity, with a scale factor of 1 on the other axis (an exact pass-through).  Entry [d, j] is
the sum of the taps of output d that read sample j after clamping, added in float32 (left to right).

Front end.  The net input of Batch_body is bf16(resize(x) - 0.5), zero padded; the reference of element (c, y, x) is

    ref = (W_y X_c W_x^T)[y, x],      mag = (|W_y| |X_c| |W_x|^T)[y, x],

in float64, X the float32 frame (uint8 frames: float32(u8) / 255 rounded once, as ToTensor divides).  The device
(prepost.cu preprocess_f32_kernel, compiled with --fmad=false) computes, with u = 2^-24:
  - per tap row i: t_i = ((v0 c0 + v1 c1) + v2 c2) + v3 c3, each product and sum rounded: a term passes through its
    product and at most 3 additions -> 4 factors (1 + d);
  - acc = ((t_0 r0 + t_1 r1) + t_2 r2) + t_3 r3 from 0 (the first addition is exact): one product and at most 3
    additions -> 4 more factors;
  - its tables hold torch's coefficients bit for bit (tests/test_batch_resize_host.py); where taps are clamped onto one
    sample the device applies them one by one while the reference's entry is their float32 sum, one rounding of a sum
    of |c| per axis -> 2 more factors;
  - /255 of uint8 frames is the same correctly rounded division the reference applies: no factor.
So |acc - ref| <= gamma_10 mag, gamma_n = n u / (1 - n u) <= 1.01 n u.  The shift rounds once more:
r = fl(acc - 0.5) lies within u |acc - 0.5| <= u (|ref - 0.5| + gamma_10 mag) of acc - 0.5.  Products of a weight and
a tiny sample may be subnormal, where a rounding errs by up to 2^-150 absolute: 2^-149 per rounding covers it.  Hence

    |r - (ref - 0.5)| <= B = 1.02 (10 u mag) + 1.01 u |ref - 0.5| + 11 * 2^-149,

and the stored element is bf16_rn(r): a round-to-nearest-even bf16 of some value in [ref - 0.5 - B, ref - 0.5 + B].
The slack (1.02, 1.01) covers gamma's denominator and the float64 rounding of the reference (~1e-15 relative).

Map side.  The per-axis operator of F.interpolate(scale_factor=8), crop to (n_h, n_w), F.interpolate(size=(H, W)) is
the float64 product S X8 of torch's float32 factors; tests/composite_ref.py's bound applies with it in place of
OpenCV's, with MAP_EXTRA_ROUNDINGS more factors: the library composes the two passes tap by tap in float64, while an
entry of S or X8 where taps are clamped onto one sample is their float32 sum, within u of the exact sum of |c|.  So an
entry of S X8 is within 2 u (|S| |X8|) of the exact composite, per axis: 4 more factors for y and x together.
"""
import numpy as np

from oracle import openpose_oracle as O

U = 2.0 ** -24
FRONT_ROUNDINGS = 10
MAP_EXTRA_ROUNDINGS = 4


def torch_matrix(n_in, n_out=None, scale_factor=None):
    """torch's float32 bicubic weights for one axis, (n_out, n_in) float64: F.interpolate(scale_factor=scale_factor),
    or size mode (n_out) when scale_factor is None."""
    import torch
    import torch.nn.functional as F
    x = torch.eye(n_in, dtype=torch.float32).reshape(n_in, 1, 1, n_in)
    with torch.no_grad():
        if scale_factor is None:
            y = F.interpolate(x, size=(1, n_out), mode="bicubic", align_corners=False)
        else:
            y = F.interpolate(x, scale_factor=(1.0, float(scale_factor)), mode="bicubic", align_corners=False)
    return y[:, 0, 0, :].T.double().numpy()


def dense(first, coef, n_in):
    """(n_out, n_in) float64 matrix of a tap table (first index, (n_out, k) float32 weights, clamped taps), duplicates
    added in float32 left to right as torch's impulse response adds them."""
    n_out, k = coef.shape
    M = np.zeros((n_out, n_in), np.float32)
    rows = np.arange(n_out)
    for j in range(k):
        idx = np.clip(np.asarray(first) + j, 0, n_in - 1)
        M[rows, idx] = M[rows, idx] + coef[:, j].astype(np.float32)
    return M.astype(np.float64)


def front_operators(H, W):
    """Batch_body's front end for an H x W frame: (h, w, W_y (h, H), W_x (w, W))."""
    scale, h, w, _, _ = O.batch_size_pad(O.BATCH_BODY_SCALE, H, W)
    return h, w, torch_matrix(H, scale_factor=scale), torch_matrix(W, scale_factor=scale)


def frames_f32(frames):
    """(n, 3, H, W) float32 frames as the reference sees them: float frames as given, uint8 (n, H, W, 3) decoded frames
    through ToTensor (float32(u8) / 255, channel order kept)."""
    f = np.asarray(frames)
    if f.dtype == np.uint8:
        return (f.astype(np.float32) / np.float32(255)).transpose(0, 3, 1, 2)
    return f.astype(np.float32)


def front_reference(x, wy, wx):
    """x (n, 3, H, W) float32 -> (ref, mag), both (n, 3, h, w) float64 (module docstring)."""
    ref = np.zeros(x.shape[:2] + (wy.shape[0], wx.shape[0]))
    mag = np.zeros_like(ref)
    for i in range(len(x)):                                  # one frame at a time: 4K frames are large in float64
        v = np.asarray(x[i], np.float64)
        ref[i] = np.matmul(np.matmul(wy, v), wx.T)
        mag[i] = np.matmul(np.matmul(np.abs(wy), np.abs(v)), np.abs(wx).T)
    return ref, mag


def front_bound(ref, mag):
    """B of the module docstring, elementwise."""
    return 1.02 * FRONT_ROUNDINGS * U * mag + 1.01 * U * np.abs(ref - 0.5) + (FRONT_ROUNDINGS + 1) * 2.0 ** -149


def bf16_rn(v):
    """nearest-even bf16 of float32 values, as float64"""
    import torch
    return torch.from_numpy(np.asarray(v, np.float32)).bfloat16().float().double().numpy()


def _round_down_f32(v):
    f = np.asarray(v, np.float64).astype(np.float32)
    return np.where(f.astype(np.float64) > v, np.nextafter(f, np.float32(-np.inf)), f)


def _round_up_f32(v):
    f = np.asarray(v, np.float64).astype(np.float32)
    return np.where(f.astype(np.float64) < v, np.nextafter(f, np.float32(np.inf)), f)


def front_check(got_bf16, ref, mag):
    """got_bf16: (n, 3, h, w) device values (float64 of bf16).  Returns (bad, ambiguous) boolean arrays: an element is
    bad when it is no bf16 rounding of any value within the bound of ref - 0.5, ambiguous when the interval straddles
    a bf16 rounding boundary (two outcomes allowed).  The interval ends are widened outwards to float32 first, so that
    rounding them to bf16 through float32 is monotone and the allowed range only grows."""
    b = front_bound(ref, mag)
    lo = bf16_rn(_round_down_f32(ref - 0.5 - b))
    hi = bf16_rn(_round_up_f32(ref - 0.5 + b))
    bad = (got_bf16 < lo) | (got_bf16 > hi)
    return bad, lo != hi


def x8_then_crop(n_net, n_resized):
    """(n_resized, n_net): F.interpolate(scale_factor=8) cropped to its first n_resized samples."""
    return torch_matrix(n_net, scale_factor=8.0)[:n_resized]


def map_operator(n_net, n_resized, n_orig):
    """per-axis operator of the map side, (n_orig, n_net) float64 product of torch's float32 factors."""
    return torch_matrix(n_resized, n_out=n_orig) @ x8_then_crop(n_net, n_resized)


def map_operators(H, W, dims):
    """dims: per scale (h, w, ho, wo) -> per scale (A_y (H, ho), A_x (W, wo)): composite_ref.axis_operators with
    torch's operator."""
    return [(map_operator(ho, h, H), map_operator(wo, w, W)) for h, w, ho, wo in dims]
