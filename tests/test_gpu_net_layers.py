"""Every launch of the CNN execution plans, layer by layer, against an fp64 convolution of the device's own input
(tests/layer_ref.py: the reference, the teacher-forced dataflow and the tolerance with its derivation).

The plans are those the pipelines build (csrc/net.cu build_net_plan), walked one step at a time through the debug entry
points (opb_net_debug_*): grouped launches of up to 8 problems with two weight sets, inputs read as channel slices of
the concat buffer, outputs written into its slices or into the fp32 final maps, the fused tails, the unfused fallback
beyond 8 problems and conv1_1 on uint8 and bf16 input.  Weights are Kaiming with random non-zero biases, and every scale
and image gets its own blurred random frame, so a tile, a bias or a weight taken from the wrong problem shows.  After
the step-wise pass the whole plan runs back to back (programmatic dependent launch overlap, one synchronisation) and must
reproduce the final maps and concat buffers bit for bit.

The expected launch forms assume a 148-SM B200 (the small-launch thresholds of conv_group / conv_pair_plan depend on the
SM count)."""
import ctypes
import time

import pytest
import torch
import torch.nn.functional as F

from oracle import openpose_oracle as O
from pytorch_openpose_b200 import _lib
from tests import layer_ref as R

pytestmark = pytest.mark.gpu

KINDS = {"body": _lib.NET_BODY, "hand": _lib.NET_HAND}
STEP_FIRST, STEP_CONV, STEP_TAIL, STEP_TAIL_WIDE, STEP_POOL = range(5)


class View(ctypes.Structure):
    _fields_ = [(f, ctypes.c_int) for f in ("n", "h", "w", "c", "cstride", "coff", "elem")]


class Step(ctypes.Structure):
    _fields_ = ([(f, ctypes.c_int) for f in ("kind", "n_problems", "block_n", "pool", "wide", "pair", "half_tiles",
                                             "weights_resident")]
                + [("name", ctypes.c_char * 64), ("layer", (ctypes.c_char * 32) * 8), ("layer2", (ctypes.c_char * 32) * 8),
                   ("scale", ctypes.c_int * 8), ("in_", View * 8), ("out", View * 8)])

    def layers(self, p):
        return self.layer[p].value.decode(), self.layer2[p].value.decode()


DTYPE = {1: torch.uint8, 2: torch.bfloat16, 4: torch.float32}

# (kind, [(n, hp, wp, in_elem)] per scale)
CONFIGS = {
    "body_4scales": ("body", [(1, 96, 128, 1), (1, 184, 248, 1), (1, 280, 376, 1), (1, 368, 496, 1)]),
    "body_2scales_batch": ("body", [(2, 184, 328, 1), (2, 368, 656, 1)]),
    "body_5scales": ("body", [(1, 48, 64, 1), (1, 96, 128, 1), (1, 144, 192, 1), (1, 192, 256, 1), (1, 240, 320, 1)]),
    "body_bf16_input": ("body", [(3, 368, 200, 2)]),
    "hand_batch": ("hand", [(8, 368, 368, 1)]),
    "hand_4scales": ("hand", [(2, 96, 96, 1), (2, 184, 184, 1), (2, 280, 280, 1), (2, 368, 368, 1)]),
}


def _weights(kind, seed):
    """Kaiming weights plus N(0, 0.1) biases, distinct per layer and branch."""
    sd = O.make_weights(kind, seed, "kaiming")
    g = torch.Generator().manual_seed(1000 + seed)
    for name in sorted(k for k in sd if k.endswith(".bias")):
        sd[name] = torch.randn(sd[name].shape, generator=g) * 0.1
    return sd


def _frames(n, hp, wp, elem, seed):
    """n blurred random frames (n, hp, wp, 3): uint8 pixels or bf16 values in [-0.5, 0.5) like the batched estimators'."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, 3, hp, wp, generator=g).cuda()
    t = torch.arange(-6, 7, dtype=torch.float32, device="cuda")
    k = torch.exp(-t * t / 8.0)
    k = k / k.sum()
    x = F.conv2d(F.pad(x, (6, 6, 0, 0), mode="reflect"), k.view(1, 1, 1, 13).repeat(3, 1, 1, 1), groups=3)
    x = F.conv2d(F.pad(x, (0, 0, 6, 6), mode="reflect"), k.view(1, 1, 13, 1).repeat(3, 1, 1, 1), groups=3)
    lo = x.amin(dim=(1, 2, 3), keepdim=True)
    hi = x.amax(dim=(1, 2, 3), keepdim=True)
    x = ((x - lo) / (hi - lo)).permute(0, 2, 3, 1).contiguous()
    if elem == 1:
        return (x * 255).round().to(torch.uint8)
    return (x - 0.5).to(torch.bfloat16)


class Plan(object):
    """One plan of a session, driven through the debug entry points."""

    def __init__(self, kind, shapes, seed=0):
        self.kind, self.shapes = kind, shapes
        self.sd = _weights(kind, seed)
        self.net = _lib.Net(KINDS[kind], self.sd)
        self.sess = self.net.session()
        arr = (ctypes.c_int * (4 * len(shapes)))(*[v for s in shapes for v in s])
        n = ctypes.c_int()
        torch.cuda.synchronize()
        _lib.check(_lib.lib().opb_net_debug_plan(self.sess.handle, len(shapes), arr, ctypes.byref(n)))
        self.n_steps = n.value
        self.info = []
        for i in range(self.n_steps):
            st = Step()
            _lib.check(_lib.lib().opb_net_debug_info(self.sess.handle, i, ctypes.byref(st)))
            self.info.append(st)

    def set_inputs(self, seed):
        self.inputs = [_frames(n, hp, wp, e, seed + 17 * s) for s, (n, hp, wp, e) in enumerate(self.shapes)]
        for s, x in enumerate(self.inputs):
            torch.cuda.synchronize()
            _lib.check(_lib.lib().opb_net_debug_set_input(self.sess.handle, s, x.data_ptr()))

    def step(self, i):
        _lib.check(_lib.lib().opb_net_debug_step(self.sess.handle, i, None))

    def run(self):
        _lib.check(_lib.lib().opb_net_debug_run(self.sess.handle))

    def read(self, i, p, which):
        v = (self.info[i].in_ if which == 0 else self.info[i].out)[p]
        t = torch.empty((v.n, v.h, v.w, v.c), dtype=DTYPE[v.elem], device="cuda")
        torch.cuda.synchronize()
        _lib.check(_lib.lib().opb_net_debug_read(self.sess.handle, i, p, which, t.data_ptr()))
        return t

    def forms(self):
        out = set()
        for st in self.info:
            if st.kind == STEP_FIRST:
                out.add("conv1_1 uint8" if st.in_[0].elem == 1 else "conv1_1 bf16")
            elif st.kind == STEP_CONV:
                if st.pair:
                    out.add("conv_tc%d pair launch, half tiles %s" % (st.block_n, "on" if st.half_tiles else "off"))
                else:
                    out.add("unfused 1x1 fallback" if self.layer_k(st.layers(0)[0]) == 1 else "conv_tc other")
                if st.wide:
                    out.add("wide conv1_2")
                if st.weights_resident:
                    out.add("resident weights")
                if len({st.layers(p)[0].rsplit("_L", 1)[-1] for p in range(st.n_problems)}) > 1:
                    out.add("two weight sets")
            elif st.kind == STEP_TAIL:
                out.add("narrow fused tail")
            elif st.kind == STEP_TAIL_WIDE:
                out.add("wide fused tail")
            if st.n_problems == 8:
                out.add("8-problem launch")
        return out

    def layer_k(self, name):
        return R.layer_table(self.kind)[name][2]


def _bits(t):
    return t.view({1: torch.uint8, 2: torch.int16, 4: torch.int32}[t.element_size()])


def _check_problem(plan, i, p, outs, worst):
    st = plan.info[i]
    kind = plan.kind
    layer, layer2 = st.layers(p)
    s = st.scale[p]
    din, dout = plan.read(i, p, 0), plan.read(i, p, 1)
    assert not torch.isnan(dout.float()).any(), "%s scale %d: NaN" % (st.name.decode(), s)
    if st.kind == STEP_POOL:
        ref = F.max_pool2d(outs[(s, layer)].float().permute(0, 3, 1, 2), 2, 2).permute(0, 2, 3, 1)
        assert torch.equal(dout.float(), ref), "maxpool after %s" % layer
        outs[(s, layer)] = dout
        return
    table = R.layer_table(kind)
    src = R.dataflow(kind)[layer]
    if src == "input":
        x_dev = plan.inputs[s]
        x_ref = R.normalise_input(x_dev)
    elif isinstance(src, tuple):
        prev = tuple(outs[(s, q)] for q in src[1])
        feat = outs[(s, src[2])]
        x_dev = R.device_concat(kind, prev, feat)
        x_ref = R.mconv1_input(kind, prev, feat)
    else:
        x_dev = outs[(s, src)]
        x_ref = x_dev
    assert torch.equal(_bits(din), _bits(x_dev.to(din.dtype))), \
        "%s (%s, scale %d): the step's input view differs from its producers' outputs" % (st.name.decode(), layer, s)
    slack = None
    if st.kind in (STEP_TAIL, STEP_TAIL_WIDE):
        _, cout, _, relu2 = table[layer2]
        w1, b1 = plan.sd[layer + ".weight"], plan.sd[layer + ".bias"]
        w2, b2 = plan.sd[layer2 + ".weight"], plan.sd[layer2 + ".bias"]
        ref, slack = R.tail_ref(x_ref, w1, b1, w2, b2, relu2)
        name = layer + "+" + layer2
        out_layer = layer2
    else:
        _, cout, _, relu = table[layer]
        ref = R.conv_ref(x_ref, plan.sd[layer + ".weight"], plan.sd[layer + ".bias"], relu, bool(st.pool))
        name, out_layer = layer, layer
    assert dout.shape[:3] == ref.shape[:3], (name, dout.shape, ref.shape)
    if dout.shape[-1] > cout:
        assert (dout[..., cout:] == 0).all(), "%s scale %d: pad channels %d.. not zero" % (name, s, cout)
    res = R.compare(dout[..., :cout], ref, R.EPS_ACC, slack)
    nonzero, spread, ok = R.not_vacuous(dout[..., :cout])
    key = name.replace("_L1", "_L*").replace("_L2", "_L*")
    w = worst.setdefault(key, [0.0, 0.0, 1.0, 1.0])
    w[0], w[1] = max(w[0], res.worst), max(w[1], res.worst_rms)
    w[2], w[3] = min(w[2], nonzero), min(w[3], spread)
    assert res.ok, "%s (%s, scale %d, problem %d of %s): %r" % (name, st.name.decode(), s, p, plan.shapes, res)
    assert ok, "%s scale %d: vacuous output (%.3f non-zero, %.3f of the channels vary)" % (name, s, nonzero, spread)
    outs[(s, out_layer)] = dout


def _cat_views(plan):
    """(step, problem) whose input view is the concat buffer, per scale."""
    cats = {}
    for i, st in enumerate(plan.info):
        for p in range(st.n_problems):
            if st.layers(p)[0].startswith("Mconv1_stage2"):
                cats.setdefault(st.scale[p], (i, p))
    return cats


def _final_views(plan):
    last = "Mconv7_stage6"
    return [(i, p) for i, st in enumerate(plan.info) for p in range(st.n_problems)
            if st.layers(p)[1].startswith(last) or st.layers(p)[0].startswith(last)]


def _print_table(title, worst):
    print("\n%s: worst |d - r| / bound per layer (element, block rms), min non-zero fraction, min varying channels" % title)
    for k, (a, b, nz, sp) in worst.items():
        print("  %-34s %.3f  %.3f  %.2f  %.2f" % (k, a, b, nz, sp))


@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_plan_layer_by_layer(config):
    kind, shapes = CONFIGS[config]
    t0 = time.time()
    plan = Plan(kind, shapes, seed=3)
    plan.set_inputs(seed=11)
    outs, worst = {}, {}
    cats = _cat_views(plan)
    pads = R.CAT_PAD[kind]
    for i, st in enumerate(plan.info):
        plan.step(i)
        for p in range(st.n_problems):
            _check_problem(plan, i, p, outs, worst)
        for s, (ci, cp) in cats.items():
            cat = plan.read(ci, cp, 0)
            for a, b in pads:
                assert (cat[..., a:b] == 0).all(), "concat pad channels %d..%d of scale %d after %s" % (a, b - 1, s,
                                                                                                       st.name.decode())
    _print_table("%s %s" % (config, shapes), worst)
    # the whole plan back to back must reproduce the step-wise final maps and concat buffers bit for bit; a run on
    # other frames first overwrites every buffer, so nothing can pass by being left over
    views = [(i, p, 1) for i, p in _final_views(plan)] + [(i, p, 0) for i, p in cats.values()]
    assert len(views) == len(shapes) * (3 if kind == "body" else 2)
    step_wise = [_bits(plan.read(*v)).clone() for v in views]
    inputs = plan.inputs
    plan.set_inputs(seed=99)
    plan.run()
    assert not all(torch.equal(_bits(plan.read(*v)), a) for v, a in zip(views, step_wise))
    plan.inputs = inputs
    for s, x in enumerate(inputs):
        _lib.check(_lib.lib().opb_net_debug_set_input(plan.sess.handle, s, x.data_ptr()))
    plan.run()
    for v, a in zip(views, step_wise):
        b = _bits(plan.read(*v))
        assert torch.equal(a, b), "step %s (%s): back-to-back run differs from the step-wise run in %d elements" % (
            plan.info[v[0]].name.decode(), "input" if v[2] == 0 else "output", int((a != b).sum()))
    print("%s: %d steps checked in %.1f s" % (config, plan.n_steps, time.time() - t0))


def test_bench_plan_conv1_1():
    """conv1_1 of the bench workload's plan (720p, scales 0.5 / 1 / 1.5 / 2, 8 frames): more 128-pixel segments than
    the grid holds, so every CTA walks across rows and images."""
    H, W = 720, 1280
    shapes = []
    for scale in (0.5, 1.0, 1.5, 2.0):
        h, w, hp, wp = (ctypes.c_int() for _ in range(4))
        _lib.check(_lib.lib().opb_scale_dims(H, W, scale, ctypes.byref(h), ctypes.byref(w), ctypes.byref(hp),
                                             ctypes.byref(wp)))
        shapes.append((8, hp.value, wp.value, 1))
    plan = Plan("body", shapes, seed=4)
    plan.set_inputs(seed=5)
    first = [i for i, st in enumerate(plan.info) if st.kind == STEP_FIRST]
    assert len(first) == 4
    segs = [n * hp * -(-wp // 128) for n, hp, wp, _ in shapes]
    assert min(segs) > 148 * 16                      # every launch walks past one pass of its grid (148 * 16 CTAs)
    worst = {}
    for i in first:
        plan.step(i)
        _check_problem(plan, i, 0, {}, worst)
    _print_table("bench plan conv1_1 %s" % shapes, worst)


def test_launch_forms_covered():
    """The configurations above reach every launch form the pipelines use."""
    forms = set()
    for config in sorted(CONFIGS):
        kind, shapes = CONFIGS[config]
        forms |= Plan(kind, shapes).forms()
    print("\nlaunch forms reached: " + "; ".join(sorted(forms)))
    need = {"conv1_1 uint8", "conv1_1 bf16", "conv_tc128 pair launch, half tiles off", "conv_tc64 pair launch, half tiles on",
            "conv_tc64 pair launch, half tiles off", "wide conv1_2", "narrow fused tail", "wide fused tail",
            "unfused 1x1 fallback", "two weight sets", "8-problem launch"}
    assert need <= forms, "not reached: %s" % sorted(need - forms)
