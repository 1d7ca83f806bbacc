"""CPU self-check of the layer-test comparison (tests/layer_ref.py): on synthetic layers, a stand-in for the device --
the same convolution summed in fp32 in another order, rounded to bf16 -- must pass, and each of the subtle kernel
defects the GPU layer tests are meant to catch, applied to the reference, must be rejected."""
import pytest
import torch
import torch.nn.functional as F

from tests import layer_ref as R

N, H, W, CIN, COUT = 2, 20, 37, 64, 32        # 37 columns: the last 16-pixel tile column holds 5 (ragged)


def _data(seed=0):
    g = torch.Generator().manual_seed(seed)
    x = R.bf16(torch.randn(N, H, W, CIN, generator=g, dtype=torch.float64) * 0.5)
    ws = [torch.randn(COUT, CIN, 3, 3, generator=g) * (2.0 / (CIN * 9)) ** 0.5 for _ in range(2)]
    bs = [torch.randn(COUT, generator=g) * 0.1 for _ in range(2)]
    return x, ws, bs


def _device(x, w, b, relu=True, store_bf16=True):
    """fp32 accumulation tap by tap in reverse order (another summation order than the fp64 reference), bf16 store."""
    k = w.shape[2]
    wq = w.to(torch.bfloat16).float()
    xp = F.pad(x.float().permute(0, 3, 1, 2), (k // 2,) * 4)
    acc = torch.zeros(x.shape[0], w.shape[0], x.shape[1], x.shape[2])
    for t in reversed(range(k * k)):
        dy, dx = divmod(t, k)
        acc += F.conv2d(xp[:, :, dy:dy + x.shape[1], dx:dx + x.shape[2]], wq[:, :, dy:dy + 1, dx:dx + 1])
    acc += b.float()[None, :, None, None]
    if relu:
        acc = torch.relu(acc)
    y = acc.permute(0, 2, 3, 1)
    return R.bf16(y) if store_bf16 else y


def test_device_stand_in_passes():
    x, ws, bs = _data()
    for w, b in zip(ws, bs):
        res = R.compare(_device(x, w, b), R.conv_ref(x, w, b, True), R.EPS_ACC)
        assert res.ok, res
        nz, spread, ok = R.not_vacuous(_device(x, w, b))
        assert ok, (nz, spread)
    # fp32 output (the final maps), no ReLU
    res = R.compare(_device(x, ws[0], bs[0], False, False), R.conv_ref(x, ws[0], bs[0], False), R.EPS_ACC)
    assert res.ok, res


def test_fused_tail_stand_in_passes():
    """A fused tail whose hidden layer is rounded from the fp32 sum: its one-ulp flips are covered by the slack of
    the reference -- and are too large for eps alone."""
    g = torch.Generator().manual_seed(3)
    x = R.bf16(torch.relu(torch.randn(4, 23, 31, 128, generator=g, dtype=torch.float64)))
    w1 = torch.randn(128, 128, 1, 1, generator=g) * (2.0 / 128) ** 0.5
    w2 = torch.randn(38, 128, 1, 1, generator=g) * (2.0 / 128) ** 0.5
    b1, b2 = torch.randn(128, generator=g) * 0.1, torch.randn(38, generator=g) * 0.1
    hidden = _device(x, w1, b1).double()
    dev = _device(hidden, w2, b2, False, False)
    ref, slack = R.tail_ref(x, w1, b1, w2, b2, False)
    flips = int((hidden != R.bf16(R.conv_ref(x, w1, b1, True))).sum())
    assert flips > 0
    res = R.compare(dev, ref, R.EPS_ACC, slack)
    assert res.ok, (res, flips)
    assert not R.compare(dev, ref, R.EPS_ACC).ok and float(slack.amax()) <= 2e-3 * float(ref.abs().amax())
    assert float(slack.mean()) <= 2e-4 * float(ref.abs().amax())        # about 1e-4 of the maximum on average


def _mutations():
    x, (w1, w2), (b1, b2) = _data(1)
    d1, d2 = _device(x, w1, b1), _device(x, w2, b2)
    r1, r2 = R.conv_ref(x, w1, b1, True), R.conv_ref(x, w2, b2, True)

    def dropped_tap():
        w = w1.clone()
        w[:, :, 0, 2] = 0                                   # tap (dy -1, dx +1) missing in one 16 x 16 tile
        r = r1.clone()
        r[1, 0:16, 16:32] = R.conv_ref(x, w, b1, True)[1, 0:16, 16:32]
        return [(d1, r)]

    def shifted_ragged_column():
        xs = torch.roll(x, 1, dims=2)                       # input read one pixel to the left ...
        r = r1.clone()
        r[:, :, 32:] = R.conv_ref(xs, w1, b1, True)[:, :, 32:]   # ... in the last (5-column) tile column only
        return [(d1, r)]

    def tile_from_other_image():
        r = r1.clone()
        r[1, 16:32, 0:16] = r1[0, 16:32, 0:16]
        return [(d1, r)]

    def tile_from_other_problem():
        r = r1.clone()
        r[0, 0:16, 16:32] = r2[0, 0:16, 16:32]
        return [(d1, r)]

    def biases_swapped():
        return [(d1, R.conv_ref(x, w1, b2, True)), (d2, R.conv_ref(x, w2, b1, True))]

    def paf_heat_swapped():
        g = torch.Generator().manual_seed(9)
        l1 = R.bf16(torch.randn(N, 12, 17, 40, generator=g, dtype=torch.float64))
        l2 = R.bf16(torch.randn(N, 12, 17, 24, generator=g, dtype=torch.float64))
        l1[..., 38:] = 0
        l2[..., 19:] = 0
        feat = R.bf16(torch.relu(torch.randn(N, 12, 17, 128, generator=g, dtype=torch.float64)))
        w = torch.randn(64, 185, 3, 3, generator=g) * (2.0 / (185 * 9)) ** 0.5
        b = torch.randn(64, generator=g) * 0.1
        dev = _device(R.mconv1_input("body", (l1, l2), feat), w, b)
        assert R.compare(dev, R.conv_ref(R.mconv1_input("body", (l1, l2), feat), w, b, True), R.EPS_ACC).ok
        swapped = torch.cat([l2[..., :19], l1[..., :38], feat], -1)
        return [(dev, R.conv_ref(swapped, w, b, True))]

    def tile_just_inside_the_bound():
        # every element of one tile off by 0.8 of its own bound: passes element by element, fails the block rms
        r = r1.clone()
        bound = R.REL * r1.abs() + R.EPS_ACC * r1.abs().amax(dim=(0, 1, 2))
        sign = torch.where(torch.arange(COUT) % 2 == 0, 1.0, -1.0).double()
        r[0, 0:16, 0:16] = d1[0, 0:16, 0:16].double() - 0.8 * bound[0, 0:16, 0:16] * sign
        res = R.compare(d1, r, R.EPS_ACC)
        assert res.worst <= 1.0, res
        return [(d1, r)]

    return {f.__name__: f for f in (dropped_tap, shifted_ragged_column, tile_from_other_image, tile_from_other_problem,
                                    biases_swapped, paf_heat_swapped, tile_just_inside_the_bound)}


@pytest.mark.parametrize("mutation", sorted(_mutations()))
def test_mutation_is_rejected(mutation):
    pairs = _mutations()[mutation]()
    results = [R.compare(d, r, R.EPS_ACC) for d, r in pairs]
    print(mutation, results)
    assert not all(res.ok for res in results), "%s passed the comparison: %s" % (mutation, results)


def test_dataflow_and_concat_layout():
    body, hand = R.dataflow("body"), R.dataflow("hand")
    assert body["conv1_1"] == "input" and body["conv2_1"] == "conv1_2" and body["conv5_1_CPM_L2"] == "conv4_4_CPM"
    assert body["Mconv1_stage2_L1"] == ("cat", ("conv5_5_CPM_L1", "conv5_5_CPM_L2"), "conv4_4_CPM")
    assert body["Mconv1_stage6_L2"] == ("cat", ("Mconv7_stage5_L1", "Mconv7_stage5_L2"), "conv4_4_CPM")
    assert hand["conv6_1_CPM"] == "conv5_3_CPM" and hand["Mconv1_stage3"] == ("cat", ("Mconv7_stage2",), "conv5_3_CPM")
    assert len(body) == len(R.layer_table("body")) and len(hand) == len(R.layer_table("hand"))
    l1, l2, feat = torch.ones(1, 1, 1, 40), 2 * torch.ones(1, 1, 1, 24), 3 * torch.ones(1, 1, 1, 128)
    ref = R.mconv1_input("body", (l1, l2), feat)
    assert ref.shape[-1] == 185 and (ref[..., :38] == 1).all() and (ref[..., 38:57] == 2).all() and (ref[..., 57:] == 3).all()
    dev = R.device_concat("body", (l1, l2), feat)
    assert dev.shape[-1] == 192 and (dev[..., :128] == 3).all() and (dev[..., 128:168] == 1).all()
    h = R.device_concat("hand", (l2,), feat)
    assert h.shape[-1] == 192 and (h[..., 128:152] == 2).all() and (h[..., 152:] == 0).all()
    assert R.mconv1_input("hand", (l2,), feat).shape[-1] == 150
