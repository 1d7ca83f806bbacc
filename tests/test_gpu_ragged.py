"""Hand()(list of square crops of any sides): one device pass (opb_hand_submit_ragged) whose row i is bit-identical to
Hand()(crops[i]) -- the per-crop geometry of the pose pipeline's ragged hand chain, fed from packed crops."""
import numpy as np
import pytest

from oracle import openpose_oracle as O

pytestmark = pytest.mark.gpu

SIDES = [1, 7, 64, 97, 150, 368, 736]
FOUR = [0.5, 1.0, 1.5, 2.0]


def _crops(sides, seed):
    import cv2
    rng = np.random.default_rng(seed)
    return [cv2.GaussianBlur(rng.integers(0, 256, (w, w, 3), dtype=np.uint8), (0, 0), 2) for w in sides]


def _hand(scales):
    from pytorch_openpose_b200 import Hand
    return Hand(O.make_weights("hand", 5, "kaiming"), scale_search=scales)


def _singles(hand, crops):
    return np.stack([hand(c) for c in crops])


@pytest.mark.parametrize("scales", [[1.0], FOUR])
def test_list_of_sides_equals_hand_on_every_crop(scales):
    hand = _hand(scales)
    crops = _crops(SIDES, 3)
    got = hand(crops)
    assert got.shape == (len(SIDES), 21, 3)
    want = _singles(hand, crops)
    for i, w in enumerate(SIDES):
        assert np.array_equal(got[i], want[i]), (scales, w)
    assert (got[:, :, 2] > 0).sum() > 10                  # key points were really found
    # replays (a captured graph from the third use on) give the same rows, also after single calls on the session
    for _ in range(3):
        assert np.array_equal(hand(crops), got)


def test_list_longer_than_one_submit_and_revisit_after_growth():
    hand = _hand([0.5, 1.0])
    rng = np.random.default_rng(11)
    long_list = _crops([int(v) for v in rng.integers(16, 220, 45)], 12)
    got = hand(long_list)                                  # two chunks of <= 32 crops over two sessions
    assert got.shape == (45, 21, 3)
    assert np.array_equal(got, _singles(hand, long_list))
    small = _crops([30, 41, 52], 13)
    first = hand(small)
    hand(_crops([9, 500, 736], 14))                       # tables and buffers grow
    assert np.array_equal(hand(small), first)              # the smaller list on the grown buffers
    assert np.array_equal(first, _singles(hand, small))


def test_equal_sides_list_is_the_stacked_batch():
    hand = _hand([0.5, 1.0])
    crops = _crops([80] * 5, 4)
    assert np.array_equal(hand(crops), hand(np.stack(crops)))


def test_crop_list_rejects_bad_crops():
    hand = _hand([1.0])
    crops = _crops([40, 50], 5)
    with pytest.raises(ValueError, match=r"Hand\(\)\(crop\)"):
        hand(crops + [np.zeros((40, 41, 3), np.uint8)])
    with pytest.raises(ZeroDivisionError):
        hand(crops + [np.zeros((0, 0, 3), np.uint8)])
    hand(crops)                                            # the session is still usable


def _abi_submit(hand, packed_ptr, offsets, where, sides, scales):
    from pytorch_openpose_b200 import _lib
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    sd = np.ascontiguousarray(sides, dtype=np.int32)
    sc, ns = _lib.scales_array(scales)
    return _lib.lib().opb_hand_submit_ragged(hand._session.handle, packed_ptr, off.ctypes.data, where, len(sd),
                                             sd.ctypes.data, sc, ns)


def test_abi_pinned_and_device_input_and_bad_arguments():
    import torch
    from pytorch_openpose_b200 import _lib
    from pytorch_openpose_b200.hand import pack_crops
    scales = [0.5, 1.0]
    hand = _hand(scales)
    crops = _crops([33, 120, 71, 200], 6)
    want = _singles(hand, crops)
    packed, offsets, sides = pack_crops(crops)
    for where in (1, 2):
        t = torch.from_numpy(packed)
        t = t.cuda() if where == 1 else t.pin_memory()
        torch.cuda.synchronize()
        _lib.check(_abi_submit(hand, t.data_ptr(), offsets, where, sides, scales))
        peaks = np.empty((len(sides), 21, 3))
        _lib.check(_lib.lib().opb_hand_wait(hand._session.handle, peaks.ctypes.data))
        assert np.array_equal(peaks, want), where
    heat = np.empty((len(sides), 22, 200, 200), np.float32)
    assert _lib.lib().opb_hand_maps(hand._session.handle, heat.ctypes.data) == _lib.OPB_ERR_INVALID
    p = packed.ctypes.data
    bad_offsets = offsets.copy()
    bad_offsets[2] += 3
    shifted = offsets + 3
    for off, sd, why in ((offsets[:1], sides[:0], "n = 0"),
                         (np.zeros(1026, np.uint64), np.ones(1025, np.int32), "n > 1024"),
                         (bad_offsets, sides, "mismatched offsets"),
                         (shifted, sides, "offsets[0] != 0"),
                         (np.zeros(2, np.uint64), np.zeros(1, np.int32), "zero side")):
        assert _abi_submit(hand, p, off, 0, sd, scales) == _lib.OPB_ERR_INVALID, why
    assert np.array_equal(hand(crops), want)               # nothing was left half-submitted
    hand(crops[1])                                         # an equal-size batch again: its maps are readable
    assert hand.last_maps(crops[1].shape).shape == (1, 120, 120, 22)


def test_list_form_leaves_the_pointer_and_pinned_forms_alone():
    """submit((device pointer, (n, h, w)), where=1) is the equal-size batch it always was; a list of different sides
    is host-only and is refused with where != 0 before anything is submitted."""
    import torch
    hand = _hand([0.5, 1.0])
    batch = np.stack(_crops([96] * 4, 7))
    want = hand(batch)
    dev = torch.from_numpy(batch).cuda()
    torch.cuda.synchronize()
    hand.submit((dev.data_ptr(), tuple(batch.shape[:3])), where=1)
    assert np.array_equal(hand.collect(), want)
    with pytest.raises(ValueError, match="where=0"):
        hand.submit(_crops([40, 50], 8), where=2)
    assert np.array_equal(hand(batch), want)


def test_pose_batch_after_a_crop_list_makes_the_hand_maps_readable_again():
    import cv2
    from pytorch_openpose_b200 import Body, _lib, motion
    hand = _hand([0.5, 1.0])
    body = Body(O.make_weights("body", 0), scale_search=[0.5])
    hand(_crops([40, 50], 9))
    heat = np.empty((2, 22, 240, 240), np.float32)         # a pose batch of one 240 x 320 frame: 2 slots of 240^2
    assert _lib.lib().opb_hand_maps(hand._session.handle, heat.ctypes.data) == _lib.OPB_ERR_INVALID
    frame = cv2.GaussianBlur(np.random.default_rng(10).integers(0, 256, (1, 240, 320, 3), dtype=np.uint8)[0], (0, 0), 2)
    est = motion.PoseEstimator(body, hand)
    pair = (body._session, hand._session)
    est.submit_batch(frame[None], pair=pair, fixed_boxes=np.array([[[10, 20, 97], [150, 30, 64]]]))
    est.collect(pair)
    _lib.check(_lib.lib().opb_hand_maps(hand._session.handle, heat.ctypes.data))
