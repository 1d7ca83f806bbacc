"""Host side of the batched hand job on the device (opb_hand_track_*), checked without a GPU: the library's box function
(the same source the device kernels run) against util.handDetect, and the tap tables of the crop resize against the
oracle's cv2 taps."""
import ctypes

import numpy as np

from oracle import openpose_oracle as O
from pytorch_openpose_b200 import _lib, util
from pytorch_openpose_b200.extract import pose_person


def _lib_boxes(pose, H, W):
    p = np.ascontiguousarray(pose, dtype=np.float64)
    out = np.zeros(8, dtype=np.int32)
    _lib.check(_lib.lib().opb_hand_track_boxes(p.ctypes.data, H, W, out.ctypes.data))
    return out.reshape(2, 4)


def _host_boxes(pose, H, W):
    """[left, right] x [x, y, w, valid] the way hand_crops_from_pose finds them; (0, 0, 0, 0) when handDetect gives none."""
    candidate, subset = pose_person(pose)
    out = np.zeros((2, 4), dtype=np.int64)
    for x, y, w, is_left in util.handDetect(candidate, subset, np.zeros((H, W, 3), np.uint8)):
        out[0 if is_left else 1] = (x, y, w, int(w > 0))
    return out


def _random_pose(rng, H, W):
    pose = np.zeros((18, 3))
    # arms may reach past every border of the frame
    pose[:, 0] = rng.uniform(-0.3 * W, 1.3 * W, 18)
    pose[:, 1] = rng.uniform(-0.3 * H, 1.3 * H, 18)
    pose[:, 2] = rng.uniform(0.05, 1.0, 18)
    kind = rng.integers(0, 6)
    if kind == 1:                                        # integer key points (what a rounded track holds)
        pose[:, :2] = np.round(pose[:, :2])
    for j in (2, 3, 4, 5, 6, 7):
        r = rng.random()
        if r < 0.1:
            pose[j] = 0                                  # missing joint
        elif r < 0.15:
            pose[j] = (3.5, -1.25, -2.25)                # present values that sum to 0: missing too
        elif r < 0.2:
            pose[j, 2] = 0.0                             # zero score but coordinates: present
    return pose


def test_box_entry_equals_handdetect_on_random_poses():
    rng = np.random.default_rng(11)
    sizes = [(1, 1), (1, 7), (5, 1), (2, 3), (17, 29), (64, 48), (240, 320), (368, 368), (480, 640), (720, 1280),
             (1280, 720)]
    n_valid = n_missing = n_tiny = 0
    for i in range(3000):
        H, W = sizes[i % len(sizes)]
        pose = _random_pose(rng, H, W)
        got, want = _lib_boxes(pose, H, W), _host_boxes(pose, H, W)
        assert np.array_equal(got, want), (i, H, W, got, want, pose[2:8])
        n_valid += int(got[:, 3].sum())
        n_missing += int((got[:, 2] == 0).sum())
        n_tiny += int((got[:, 2] == 1).sum())
    assert n_valid > 1000 and n_missing > 500 and n_tiny > 10


def test_box_entry_edge_cases():
    H, W = 240, 320

    def arm(shoulder, elbow, wrist, side="right"):
        pose = np.zeros((18, 3))
        js = (2, 3, 4) if side == "right" else (5, 6, 7)
        for j, (x, y) in zip(js, (shoulder, elbow, wrist)):
            pose[j] = (x, y, 0.5)
        return pose

    cases = [
        arm((100, 50), (100, 90), (100, 130)),                     # reach 40 > 0.9 * upper 36
        arm((100, 50), (100, 100), (100, 145)),                    # reach 45 == 0.9 * 50: a tie in max()
        arm((0, 0), (30, 40), (57, 76)),                           # 45 == 0.9 * 50 again, diagonal
        arm((310, 10), (318, 5), (319.9, 0.5)),                    # leaves at the top right corner: width 0 or 1
        arm((10, 230), (2, 236), (0.2, 239.7)),                    # bottom left corner
        arm((300, 120), (315, 120), (319.5, 120)),                 # right border: clipped to width 0..1
        arm((160, 120), (160, 121), (160, 122)),                   # tiny box
        arm((160, 120), (170, 120), (400, 120)),                   # wrist outside: x > W, width < 0
        arm((160, 120), (170, 120), (180, 120), "left"),
    ]
    for x in np.linspace(316, 321, 101):                           # widths clipped to 0 and 1 at the right border
        cases.append(arm((x - 20, 100), (x - 10, 100), (x, 100)))
        cases.append(arm((x - 2, 100), (x - 1, 100), (x, 100)))
    for pose in cases:
        assert np.array_equal(_lib_boxes(pose, H, W), _host_boxes(pose, H, W)), pose[2:8]
    widths = {int(_lib_boxes(p, H, W)[:, 2].max()) for p in cases}
    assert 0 in widths and 1 in widths
    # a tie: max(reach, 0.9 * upper) with equal values
    a = arm((100, 50), (100, 100), (100, 145))
    assert np.sqrt(45.0 ** 2) == 0.9 * np.sqrt(50.0 ** 2)
    assert _lib_boxes(a, H, W)[1, 2] == _host_boxes(a, H, W)[1, 2] > 0


def _track_taps(side, boxsize):
    first = np.zeros(boxsize, dtype=np.int32)
    coef = np.zeros((boxsize, 4), dtype=np.float32)
    _lib.check(_lib.lib().opb_debug_hand_track_taps(side, boxsize, first.ctypes.data, coef.ctypes.data))
    return first, coef


def test_track_taps_are_cv2_dsize_taps():
    """The tables of the crop resize use cv2's dsize-mode step 1 / (boxsize / side); for boxsize 368 they are the
    ragged tables of the pose pipeline at hand scale 1.0."""
    for boxsize in (368, 184):
        for side in range(1, 1501):
            first, coef = _track_taps(side, boxsize)
            of, oc = O.cubic_taps(side, boxsize, 1.0 / (boxsize / side))
            assert np.array_equal(first, of) and np.array_equal(coef.view(np.uint32), oc.astype(np.float32).view(np.uint32)), (side, boxsize)
            if boxsize == 368:
                h, w, hp, wp = (ctypes.c_int() for _ in range(4))
                _lib.check(_lib.lib().opb_scale_dims(side, side, 1.0, ctypes.byref(h), ctypes.byref(w), ctypes.byref(hp),
                                                     ctypes.byref(wp)))
                assert w.value == 368
                rf = np.zeros(368, dtype=np.int32)
                rc = np.zeros((368, 4), dtype=np.float32)
                _lib.check(_lib.lib().opb_debug_resize_taps(side, 368, 1.0 / (1.0 * 368.0 / side), rf.ctypes.data,
                                                            rc.ctypes.data))
                assert np.array_equal(first, rf) and np.array_equal(coef.view(np.uint32), rc.view(np.uint32)), side
