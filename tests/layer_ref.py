"""Layer-by-layer reference of the CNN execution plans, and the comparison the layer tests apply.

The reference of one convolution is an fp64 convolution (`F.conv2d` in float64) of the device's own bf16 input with the
weights rounded to bf16, as the device holds them (conv1_1's fp32 `w_first` table holds bf16-rounded values too), plus
the fp32 bias, ReLU and 2x2 max-pool as in `src/model.py`.  A fused tail's hidden layer is `bf16(relu(conv1))`: exactly
what the unfused path would store between the two 1x1 layers.

Teacher forcing: the input of a layer is built from the DEVICE outputs of the layers that produce it, following the
reference's dataflow (`oracle.openpose_oracle.body_layers` / `hand_layers`): each layer reads its predecessor, the first
layer of a stage reads the trunk features, `Mconv1` reads `torch.cat([L1, L2, feat])` (hand: `[out, feat]`) in the
reference's channel order with the checkpoint's unpermuted weights.  The device's own input view is checked separately
against the same producers in the device's concat layout, so the concat layout and the Mconv1 weight permutation are
both under test.

Comparison, per element of each problem:  |d - r| <= 2^-8 |r| + eps * max|r|, the max taken per output channel.

* 2^-8 |r| is the bf16 rounding of the stored output: a bf16 keeps 8 significant bits, so rounding to nearest moves a
  value by at most half an ulp, 2^-8 of its magnitude.
* eps * max|r| is the fp32 accumulation.  A sum of K products accumulated in fp32 with round-to-nearest carries an
  error that grows like a random walk, about u * sqrt(K) of the partial sums (u = 2^-24); tensor cores may align and
  truncate in their internal additions, which biases the error, so it can grow linearly: up to K * u of the partial
  sums.  The deepest layers have K = 7 * 7 * 192 = 9408 (Mconv1): K * u = 5.6e-4, and the partial sums stay within a
  small multiple of the channel's largest output.  EPS_ACC = 2^-10 = 9.8e-4 covers that.  (At 2^-12 one element of an
  Mconv1 launch reached 1.13 of its bound, block rms 0.64: an element whose bf16 rounding used its whole half-ulp
  allowance, with the accumulation error on top.  At 2^-10 the worst element of every configuration of
  tests/test_gpu_net_layers.py is 0.96 of its bound.)  That is still 2x tighter than the 2e-3 of tests/test_gpu_conv.py,
  and per output channel instead of over the whole output.
* A fused tail rounds its hidden layer to bf16 on the device as the reference does, but from an fp32 sum that differs
  from the fp64 one by the error above.  Where the exact hidden value lies that close to a bf16 rounding boundary, the
  two roundings differ by one ulp (2^-8 to 2^-7 of the value), and that flip reaches every output of the pixel through
  one weight of the second layer.  It cannot be budgeted inside eps: a single flip of a hidden value 3.6 times its
  rms, through a weight of 1.7 sigma, already moves an output by 1.04e-3 of its channel's maximum (tests/
  test_layer_ref.py), and larger maps meet larger combinations.  So the reference of a tail carries the flips
  explicitly (`tail_ref`): a hidden value is ambiguous when it lies within 16 u sqrt(K1) max|hidden| of a rounding
  midpoint (16 times the random-walk error of its K1-term sum, above the linear bound K1 * u for K1 = 128), and each output element gets the slack
  sum over its ambiguous hidden values of |w2| * ulp.  A few % of the hidden values are ambiguous; the slack is about
  1e-4 of the maximum on average and reaches the 1e-3 level only where a large hidden value meets a large weight.  eps
  stays EPS_ACC for every layer.

A second check works on blocks of (problem, 16 x 16 output pixels, 16 channels): the rms of d - r must stay below
2^-8 rms(r) * sqrt(1/3 + 1.2 / sqrt(k)) + eps / 2 * max|r| + rms(slack) (k elements in the block, max over its
channels).  Rounding errors spread uniformly over +-half an ulp have an rms of 1/sqrt(3) of their bound (the 1.2 / sqrt(k) term is four
standard deviations of the mean square of k such errors), so a tile whose every element is off by just under the
per-element bound -- a wrong bias, a stale value rounded differently -- fails here although each element passes."""
import math

import torch
import torch.nn.functional as F

REL = 2.0 ** -8
EPS_ACC = 2.0 ** -10
U = 2.0 ** -24
BLOCK = 16

# pad channels of the views the last layer of a stage writes (real channels, view channels)
REAL_OUT = {"paf": (38, 40), "heat": (19, 24), "hand": (22, 24)}
# channels of the 192-channel concat buffer that no layer may ever make non-zero
CAT_PAD = {"body": [(166, 168), (187, 192)], "hand": [(150, 192)]}


def bf16(t):
    """t rounded to bf16, in t's dtype."""
    return t.to(torch.bfloat16).to(t.dtype)


def conv_ref(x_nhwc, weight, bias, relu, pool=False):
    """fp64 convolution of x (n, h, w, cin) with bf16-rounded OIHW `weight` and fp32 `bias`, stride 1, same padding;
    ReLU and 2x2/2 max-pool as src/model.py.  Returns (n, h', w', cout) float64 on x's device."""
    x = x_nhwc.double().permute(0, 3, 1, 2)
    w = weight.to(torch.bfloat16).double().to(x.device)
    b = bias.float().double().to(x.device)
    y = F.conv2d(x, w, b, 1, weight.shape[2] // 2)
    if relu:
        y = torch.relu(y)
    if pool:
        y = F.max_pool2d(y, 2, 2)
    return y.permute(0, 2, 3, 1)


def tail_ref(x_nhwc, w1, b1, w2, b2, relu2):
    """A fused 1x1 -> ReLU -> 1x1 tail: the hidden layer is rounded to bf16 as the unfused path would store it.
    Returns (reference, slack): slack bounds, per output element, what one-ulp flips of the ambiguous hidden values
    (those within the fp32 accumulation error of a bf16 rounding midpoint) can move it."""
    h = conv_ref(x_nhwc, w1, b1, True)
    hb = bf16(h)
    mag = h.abs()
    ulp = torch.where(mag > 0, torch.exp2(torch.floor(torch.log2(mag.clamp_min(1e-300))) - 7), torch.zeros_like(h))
    delta = 16 * U * math.sqrt(w1.shape[1]) * mag.amax(dim=(0, 1, 2))
    ambiguous = (ulp / 2 - (h - hb).abs()) <= delta
    slack = conv_ref(torch.where(ambiguous, ulp, torch.zeros_like(ulp)), w2.abs(), torch.zeros(w2.shape[0]), False)
    return conv_ref(hb, w2, b2, relu2), slack


def normalise_input(x):
    """conv1_1's input as the kernel sees it: uint8 pixels -> x / 256 - 0.5 (exact in bf16), bf16 values as they are."""
    if x.dtype == torch.uint8:
        return x.double() / 256.0 - 0.5
    return x.double()


def mconv1_input(kind, prev, feat):
    """The input of a refinement stage in the reference's channel order: cat([L1, L2, feat]) (src/model.py:112) for
    the body, cat([out, feat]) (src/model.py:200) for the hand.  `prev`: the views the previous stage wrote (PAF 40 /
    heat 24 channels, hand 24), of which the first 38 / 19 / 22 are real."""
    if kind == "body":
        l1, l2 = prev
        return torch.cat([l1[..., :38], l2[..., :19], feat[..., :128]], -1)
    (out,) = prev
    return torch.cat([out[..., :22], feat[..., :128]], -1)


def device_concat(kind, prev, feat):
    """The 192-channel concat buffer as the device lays it out (net.cu):  body [feat | PAF 38 + 2 zero | heat 19 + 5
    zero], hand [feat | heat 22 + 2 zero | 40 zero]."""
    if kind == "body":
        l1, l2 = prev
        return torch.cat([feat, l1, l2], -1)
    (out,) = prev
    pad = torch.zeros(out.shape[:-1] + (40,), dtype=out.dtype, device=out.device)
    return torch.cat([feat, out, pad], -1)


class Result(object):
    """Outcome of `compare`: worst per-element and per-block normalised errors (<= 1 passes)."""

    def __init__(self, worst, worst_rms, where, nan):
        self.worst, self.worst_rms, self.where, self.nan = worst, worst_rms, where, nan

    @property
    def ok(self):
        return not self.nan and self.worst <= 1.0 and self.worst_rms <= 1.0

    def __repr__(self):
        return "worst %.3f (at %s), worst block rms %.3f%s" % (self.worst, self.where, self.worst_rms,
                                                               ", NaN" if self.nan else "")


def _blocks(t, b=BLOCK):
    """Sum of t (n, h, w, c) over blocks of b x b pixels and b channels (zero-padded at the edges)."""
    n, h, w, c = t.shape
    t = F.pad(t, (0, -c % b, 0, -w % b, 0, -h % b))
    n, h, w, c = t.shape
    return t.reshape(n, h // b, b, w // b, b, c // b, b).sum(dim=(2, 4, 6))


def compare(d, r, eps=EPS_ACC, slack=None, rel=REL):
    """d: the device result, r: the fp64 reference, both (n, h, w, c) of ONE problem; slack: an extra per-element
    allowance of the reference (a fused tail's flips).  Returns a Result."""
    d = d.double()
    r = r.double().to(d.device)
    assert d.shape == r.shape, (d.shape, r.shape)
    slack = torch.zeros_like(r) if slack is None else slack.double().to(d.device)
    nan = bool(torch.isnan(d).any())
    err = (d - r).abs()
    cmax = r.abs().amax(dim=(0, 1, 2))                                   # per output channel
    bound = rel * r.abs() + eps * cmax + slack
    norm = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))
    flat = int(torch.argmax(torch.nan_to_num(norm, nan=math.inf)))
    n, h, w, c = d.shape
    where = (flat // (h * w * c), flat // (w * c) % h, flat // c % w, flat % c)
    worst = float(norm.reshape(-1)[flat]) if not nan else math.inf
    ones = torch.ones_like(r)
    k = _blocks(ones)
    ms_err = _blocks(err * err) / k
    ms_ref = _blocks(r * r) / k
    gmax = F.pad(cmax, (0, -c % BLOCK)).reshape(-1, BLOCK).amax(1)        # per channel group
    rms_bound = rel * ms_ref.sqrt() * torch.sqrt(1.0 / 3.0 + 1.2 / k.sqrt()) + 0.5 * eps * gmax + (_blocks(slack * slack) / k).sqrt()
    rms_norm = torch.where(rms_bound > 0, ms_err.sqrt() / rms_bound.clamp_min(1e-300),
                           torch.where(ms_err > 0, math.inf, 0.0))
    worst_rms = float(torch.nan_to_num(rms_norm, nan=math.inf).max())
    return Result(worst, worst_rms, where, nan)


def not_vacuous(d, min_nonzero=0.03, min_spread=0.25):
    """(fraction of non-zero elements, fraction of channels that are not constant, ok); a check counts only when the
    device output has real structure: at least `min_nonzero` non-zero elements and `min_spread` of the channels varying.
    (Deep in the network a small map is nearly uniform, and a ReLU layer then switches every channel whose mean is
    negative off at every pixel: a fraction of the channels, not every channel, must vary.)"""
    d = d.float()
    nonzero = float((d != 0).float().mean())
    c = d.shape[-1]
    flat = d.reshape(-1, c)
    spread = float((flat.amax(0) > flat.amin(0)).float().mean())
    return nonzero, spread, nonzero >= min_nonzero and spread >= min_spread


def dataflow(kind):
    """{layer: producer} of the reference network: the predecessor layer's name, "input" for conv1_1, and for the first
    layer of a refinement stage the tuple ("cat", previous stage's last layers, trunk's last layer)."""
    from oracle import openpose_oracle as O
    blocks = O.body_layers() if kind == "body" else O.hand_layers()
    layers = {blk: [l for l in ls if l != "pool"] for blk, ls in blocks}
    head = "model0" if kind == "body" else "model1_0"
    feat = layers[head][-1][0]
    pred = {}
    for blk, ls in blocks:
        ls = [l for l in ls if l != "pool"]
        for j, l in enumerate(ls):
            if j > 0:
                pred[l[0]] = ls[j - 1][0]
            elif blk == head:
                pred[l[0]] = "input"
            elif blk in ("model1_1", "model1_2"):
                pred[l[0]] = feat
            elif kind == "body":
                s = int(blk[5:blk.index("_")])
                prev = tuple(layers["model%d_%d" % (s - 1, b)][-1][0] if s > 2 else layers["model1_%d" % b][-1][0]
                             for b in (1, 2))
                pred[l[0]] = ("cat", prev, feat)
            else:
                s = int(blk[5:])
                prev = layers["model%d" % (s - 1)][-1][0] if s > 2 else layers["model1_1"][-1][0]
                pred[l[0]] = ("cat", (prev,), feat)
    return pred


def layer_table(kind):
    """{layer: (cin, cout, k, relu)} of the reference network."""
    from oracle import openpose_oracle as O
    blocks = O.body_layers() if kind == "body" else O.hand_layers()
    return {l[0]: l[1:] for _, ls in blocks for l in ls if l != "pool"}
