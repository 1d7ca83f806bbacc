"""Host side of Hand()(list of crops): which lists take the ragged path, and the packed layout and validation that
opb_hand_submit_ragged reads."""
import numpy as np
import pytest

from pytorch_openpose_b200.hand import _is_ragged, crop_sides, pack_crops


def test_only_lists_of_different_shapes_are_ragged():
    a, b = np.zeros((5, 5, 3), np.uint8), np.zeros((6, 6, 3), np.uint8)
    assert _is_ragged([a, b]) and _is_ragged((b, a, a))
    assert not _is_ragged([a, a])                           # stacks to the equal-size batch it always was
    assert not _is_ragged(np.stack([a, a]))
    assert not _is_ragged(a)


def test_pack_layout():
    rng = np.random.default_rng(0)
    sides = [1, 7, 3, 64, 2]
    crops = [rng.integers(0, 256, (w, w, 3), dtype=np.uint8) for w in sides]
    crops[2] = crops[2].astype(np.int64)                    # converted like the equal-size path converts
    crops[3] = np.asfortranarray(crops[3])                  # any memory order
    packed, offsets, got_sides = pack_crops(crops)
    assert packed.dtype == np.uint8 and offsets.dtype == np.uint64 and got_sides.dtype == np.int32
    assert list(got_sides) == sides
    assert offsets[0] == 0 and len(offsets) == len(sides) + 1
    assert list(np.diff(offsets)) == [3 * w * w for w in sides]
    assert offsets[-1] == packed.size
    for i, c in enumerate(crops):
        assert np.array_equal(packed[offsets[i]:offsets[i + 1]].reshape(c.shape), c.astype(np.uint8)), i


def test_crop_validation():
    ok = np.zeros((4, 4, 3), np.uint8)
    with pytest.raises(ValueError, match=r"Hand\(\)\(crop\)"):
        crop_sides([ok, np.zeros((4, 5, 3), np.uint8)])
    with pytest.raises(ValueError, match="crop 1"):
        crop_sides([ok, np.zeros((4, 4), np.uint8)])
    with pytest.raises(ValueError):
        crop_sides([ok, np.zeros((4, 4, 4), np.uint8)])
    with pytest.raises(ZeroDivisionError):                  # what Hand()(crop) raises on an empty crop
        crop_sides([ok, np.zeros((0, 3, 3), np.uint8)])
    assert list(crop_sides([ok, [[[1, 2, 3]]]])) == [4, 1]  # nested lists are crops too


def test_list_of_different_sides_is_host_only():
    from pytorch_openpose_b200.hand import Hand
    hand = Hand.__new__(Hand)                               # no network: the check comes before anything is submitted
    hand.scale_search = [1.0]
    hand._session = None
    with pytest.raises(ValueError, match="where=0"):
        hand.submit([np.zeros((4, 4, 3), np.uint8), np.zeros((5, 5, 3), np.uint8)], where=2)
