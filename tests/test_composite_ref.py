"""CPU checks of tests/composite_ref.py: a float32 stand-in of the device's composite chains passes the float64 bound,
and each of four small defects of that arithmetic is rejected by it."""
import numpy as np
import pytest

from oracle import openpose_oracle as O
from tests import composite_ref as R


def _case(H, W, scales, seed, C=3):
    plan = O.scale_plan(H, W, scales)
    dims = [(p["h"], p["w"], p["ho"], p["wo"]) for p in plan]
    rng = np.random.default_rng(seed)
    # positive, smooth-ish net outputs (like heat maps): no cancellation to hide a defect behind
    nets = [(0.5 + rng.random((ho, wo, C))).astype(np.float32) for _, _, ho, wo in dims]
    return nets, R.axis_operators(H, W, dims)


@pytest.mark.parametrize("H,W,scales", [(97, 131, (0.5,)), (120, 160, (0.5, 1.0)), (64, 88, (0.5, 0.75, 1.0)),
                                        (240, 320, (0.25, 0.5))])
def test_float32_standin_is_within_bound(H, W, scales):
    nets, ops = _case(H, W, scales, 1)
    assert R.excess(R.standin(nets, ops), nets, ops) <= 1.0
    # large dynamic range: one sample of 1e4 among O(0.1) values, the bound follows the magnitudes element-wise
    big = [n.copy() for n in nets]
    big[0][big[0].shape[0] // 2, big[0].shape[1] // 2, 0] = 1e4
    big = [(0.1 * n).astype(np.float32) for n in big]
    assert R.excess(R.standin(big, ops), big, ops) <= 1.0


def _dropped_tap(kind, s, t):
    if kind == "x" and s == 0:
        f, w = t[0], t[1].copy()
        o = len(f) // 2
        w[o, np.argmax(np.abs(w[o]))] = 0
        return f, w
    return t


def _neighbour_row(kind, s, t):
    if kind == "row" and s == 0:
        rows = t.copy()
        y = len(rows) // 3
        rows[y, 2] = min(rows[y, 2] + 1, rows.max())
        return rows
    return t


def _missing_fold(kind, s, t):
    if kind == "fold" and s == 1:
        return np.float32(1)
    return t


def _weight_off(kind, s, t):
    if kind == "y" and s == 0:
        f, w = t[0], t[1].copy()
        o = len(f) // 2
        j = np.argmax(np.abs(w[o]))
        w[o, j] = np.float32(np.float64(w[o, j]) * (1 + 2.0 ** -16))
        return f, w
    return t


@pytest.mark.parametrize("mutate", [_dropped_tap, _neighbour_row, _missing_fold, _weight_off],
                         ids=["dropped_tap", "neighbour_row", "missing_fold", "weight_off_2^-16"])
def test_bound_rejects_defects(mutate):
    nets, ops = _case(120, 160, (0.5, 1.0), 2)
    assert R.excess(R.standin(nets, ops), nets, ops) <= 1.0
    assert R.excess(R.standin(nets, ops, mutate), nets, ops) > 1.0


@pytest.mark.parametrize("H,W,scales,mode,fused", [(368, 656, (1.0,), 0, 1), (720, 1280, (0.5, 1.0, 1.5, 2.0), 0, 1),
                                                   (97, 131, (0.5,), 0, 1), (97, 131, (0.5, 1.5), 0, 0),
                                                   (40, 40, (2.0,), 0, 0), (720, 1280, (0.5,), 1, 1),
                                                   (200, 33, (0.5,), 1, 1)])
def test_debug_post_dims(H, W, scales, mode, fused):
    """opb_body_debug_post_dims (host only): the net output sizes of the plan a Body / Batch_body call builds, and
    whether its heat maps go through the fused peak kernel"""
    import ctypes
    from pytorch_openpose_b200 import _lib
    sc, ns = _lib.scales_array(scales)
    hw = (ctypes.c_int * (2 * ns))()
    f = ctypes.c_int()
    _lib.check(_lib.lib().opb_body_debug_post_dims(H, W, sc, ns, mode, hw, ctypes.byref(f)))
    if mode == 0:
        want = [(p["ho"], p["wo"]) for p in O.scale_plan(H, W, scales)]
    else:
        _, h, w, ph, pw = O.batch_size_pad(scales[0], H, W)
        want = [((h + ph) // 8, (w + pw) // 8)]
    assert [(hw[2 * i], hw[2 * i + 1]) for i in range(ns)] == want
    assert f.value == fused
    with pytest.raises(_lib.OpbError):
        sc2, _ = _lib.scales_array((0.5, 1.0))
        _lib.check(_lib.lib().opb_body_debug_post_dims(H, W, sc2, 2, 1, hw, ctypes.byref(f)))     # Batch_body: one scale
