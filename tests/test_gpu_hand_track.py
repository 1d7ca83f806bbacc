"""The batched hand job on the device (Batch_hand.submit_track / track, opb_hand_track_*) against the host composition it
replaces: extract.hand_crops_from_pose -> Batch_hand on the left and on the right crops -> extract._box_to_roi
(srcmx/Batch_motion_Estimation.py:19-63)."""
import contextlib

import numpy as np
import pytest

from oracle import openpose_oracle as O
from pytorch_openpose_b200 import util
from pytorch_openpose_b200.extract import _box_to_roi, hand_crops_from_pose, pose_person

pytestmark = pytest.mark.gpu


@contextlib.contextmanager
def _cv2_optimized(on):
    """IPP's cubic resize differs from OpenCV's own arithmetic by 1 LSB on some pixels; the device implements the latter."""
    import cv2
    old = cv2.useOptimized()
    cv2.setUseOptimized(on)
    try:
        yield
    finally:
        cv2.setUseOptimized(old)


def _frames(n, H, W, seed):
    import cv2
    rng = np.random.default_rng(seed)
    return np.stack([cv2.GaussianBlur(rng.integers(0, 256, (H, W, 3), dtype=np.uint8), (0, 0), 2) for _ in range(n)])


def _poses(n, H, W, seed):
    """Random arms, mostly inside the frame, some leaving it; some joints missing.  A box of width 0 (the host path's
    cv2.resize raises on it) is turned into a missing hand by dropping that wrist."""
    rng = np.random.default_rng(seed)
    poses = np.zeros((n, 18, 3))
    for f in range(n):
        p = poses[f]
        p[:, 0] = rng.uniform(-0.1 * W, 1.1 * W, 18)
        p[:, 1] = rng.uniform(-0.1 * H, 1.1 * H, 18)
        p[:, 2] = rng.uniform(0.1, 1.0, 18)
        for j in (2, 3, 4, 5, 6, 7):
            if rng.random() < 0.08:
                p[j] = 0
        candidate, subset = pose_person(p)
        for x, y, w, is_left in util.handDetect(candidate, subset, np.zeros((H, W, 3), np.uint8)):
            if w <= 0:
                p[7 if is_left else 4] = 0
    return poses


def _host(est, frames, poses, boxsize=368):
    """HandMat of the host path and its crops (left, right)."""
    items = [hand_crops_from_pose(frames[f], poses[f], boxsize) for f in range(len(frames))]
    lefts = np.stack([it[0] for it in items])
    rights = np.stack([it[2] for it in items])
    mats = np.zeros((len(frames), 42, 3))
    for lo in range(0, len(frames), 32):
        est.submit_frames(lefts[lo:lo + 32])
        L = est.collect()
        est.submit_frames(rights[lo:lo + 32])
        R = est.collect()
        for i in range(len(L)):
            mats[lo + i, 21:] = _box_to_roi(R[i], items[lo + i][3], boxsize, mirrored=False)
            mats[lo + i, :21] = _box_to_roi(L[i], items[lo + i][1], boxsize, mirrored=True)
    return mats, lefts, rights


@pytest.fixture(scope="module")
def est():
    from pytorch_openpose_b200 import Batch_hand
    return Batch_hand(O.make_weights("hand", 5, "kaiming"))


def test_crops_equal_host_crops(est):
    H, W = 240, 320
    frames = _frames(8, H, W, 1)
    poses = _poses(8, H, W, 2)
    poses[1, 5:8] = 0                                            # no left hand
    poses[2, 2:5] = 0                                            # no right hand
    poses[3, 2:8] = 0                                            # no hands
    poses[4, 2:5] = [(280, 200, 0.5), (300, 220, 0.5), (318, 238, 0.5)]       # right hand at the bottom right border
    poses[4, 5:8] = [(40, 30, 0.5), (20, 15, 0.5), (3, 2, 0.5)]               # left hand at the top left border
    est.submit_track(frames, poses)
    got = est.track_crops()
    est.collect_track()
    with _cv2_optimized(False):
        _, lefts, rights = _host(est, frames, poses)
    assert np.array_equal(got[0::2], lefts) and np.array_equal(got[1::2], rights)
    assert (got[2] == 128).all() and (got[5] == 128).all() and (got[6] == 128).all() and (got[7] == 128).all()
    assert not (got[8] == 128).all() and not (got[9] == 128).all()
    with _cv2_optimized(True):
        _, lefts, rights = _host(est, frames, poses)
    assert np.abs(got[0::2].astype(int) - lefts).max() <= 1 and np.abs(got[1::2].astype(int) - rights).max() <= 1


def test_handmat_equals_host_path(est):
    mats = []
    with _cv2_optimized(False):
        for (H, W), n, seed in (((240, 320), 150, 3), ((720, 1280), 40, 4), ((96, 72), 20, 5)):
            frames = _frames(n, H, W, seed)
            poses = _poses(n, H, W, seed + 100)
            poses[:5, 2:8] = 0                                   # frames without hands
            poses[5:8, 5:8] = 0                                  # one hand only
            got = est.track(frames, poses)
            ref, _, _ = _host(est, frames, poses)
            assert got.shape == (n, 42, 3)
            assert np.array_equal(got, ref), (H, W, np.argwhere(got != ref)[:5])
            mats.append(got)
    allm = np.concatenate(mats)
    assert len(allm) >= 200
    # frames without hands: coordinates 0, but the scores Batch_hand finds on the grey crops (not zeros)
    est.submit_frames(np.full((1, 368, 368, 3), 128, np.uint8))
    grey = est.collect()[0]
    assert (allm[:5, :, :2] == 0).all()
    assert np.array_equal(allm[:5, :21, 2], np.broadcast_to(grey[:, 2], (5, 21)))
    assert np.array_equal(allm[:5, 21:, 2], np.broadcast_to(grey[:, 2], (5, 21)))
    assert (allm[:, :21, 2] > 0).any() and (allm[:, 21:, 2] > 0).any()


def test_batch_size_does_not_change_rows(est):
    H, W = 240, 320
    frames = _frames(32, H, W, 7)
    poses = _poses(32, H, W, 8)
    rows = []
    for n in (1, 7, 32):
        est.submit_track(frames[32 - n:], poses[32 - n:])
        rows.append(est.collect_track()[-1])
    assert np.array_equal(rows[0], rows[1]) and np.array_equal(rows[0], rows[2])


def test_graph_replay_and_growing_frames(est):
    from pytorch_openpose_b200 import _lib
    s = est.net.session()
    H, W = 120, 160
    frames = _frames(6, H, W, 9)
    poses = _poses(6, H, W, 10)
    outs = []
    for _ in range(5):                                          # the third use on is a CUDA graph
        est.submit_track(frames, poses, s)
        outs.append(est.collect_track(s))
    assert all(np.array_equal(o, outs[0]) for o in outs[1:])
    with _cv2_optimized(False):
        assert np.array_equal(outs[0], _host(est, frames, poses)[0])
        big = _frames(6, 360, 480, 11)                           # tables regrow, the frame buffer moves
        bposes = _poses(6, 360, 480, 12)
        for _ in range(4):
            est.submit_track(big, bposes, s)
            out = est.collect_track(s)
            assert np.array_equal(out, _host(est, big, bposes)[0])
        for _ in range(2):                                       # and back to the small frames
            est.submit_track(frames, poses, s)
            assert np.array_equal(est.collect_track(s), outs[0])
    import torch                                                # frames already on the device
    est.submit_track(torch.from_numpy(frames).cuda(), poses, s)
    assert np.array_equal(est.collect_track(s), outs[0])
    with pytest.raises(ValueError):
        est.submit_track(frames, poses[:5], s)
    with pytest.raises(_lib.OpbError):
        _lib.check(_lib.lib().opb_hand_track_submit(s.handle, frames.ctypes.data, 0, 6, H, W, poses.ctypes.data, 100))


def test_default_init_weights():
    from pytorch_openpose_b200 import Batch_hand
    e = Batch_hand(O.make_weights("hand", 0))
    frames = _frames(5, 200, 300, 13)
    poses = _poses(5, 200, 300, 14)
    with _cv2_optimized(False):
        assert np.array_equal(e.track(frames, poses, boxsize=184), _host(e, frames, poses, 184)[0])


def _track_video(path, n, w, h):
    import cv2
    wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (w, h))
    assert wr.isOpened()
    rng = np.random.default_rng(21)
    for _ in range(n):
        wr.write(cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), 3))
    wr.release()


def _pose_track(n):
    """A person with both arms moving from frame to frame (ROI coordinates of a 288 x 224 ROI)."""
    mats = np.zeros((n, 18, 3))
    for k in range(n):
        joints = {1: (144, 50), 2: (120, 60), 3: (100 + k % 7, 100), 4: (90 + 2 * (k % 5), 150 + k % 9),
                  5: (170, 60), 6: (190 - k % 6, 100), 7: (205 - 2 * (k % 4), 150 + k % 8)}
        for j, (x, y) in joints.items():
            mats[k, j] = (x, y, 0.8)
    return mats


@pytest.mark.parametrize("workers", [1, 2])
def test_job_equals_host_path(tmp_path, monkeypatch, est, workers):
    import joblib
    from pytorch_openpose_b200 import extract
    path = str(tmp_path / "v.avi")
    _track_video(path, 11, 320, 240)
    rec = [(16, 8), (304, 232)]
    track = _pose_track(11)
    dev = extract.batch_hand_extraction(path, track, rec, str(tmp_path / "d.pkl"), est, batchsize=4, log=lambda m: None,
                                        decode_workers=workers, sessions=2)
    monkeypatch.setenv("OPB_HOST_HANDS", "1")
    with _cv2_optimized(False):
        host = extract.batch_hand_extraction(path, track, rec, str(tmp_path / "h.pkl"), est, batchsize=4,
                                             log=lambda m: None)
    monkeypatch.delenv("OPB_HOST_HANDS")
    assert dev.shape == (11, 42, 3)
    assert np.array_equal(joblib.load(str(tmp_path / "d.pkl")), dev)
    assert np.array_equal(joblib.load(str(tmp_path / "h.pkl")), host)
    assert np.array_equal(dev, host)
    assert (dev[:, :21, 2] > 0).any() and (dev[:, 21:, 2] > 0).any()        # both hands were really estimated
    with pytest.raises(AssertionError):
        extract.batch_hand_extraction(path, track[:10], rec, str(tmp_path / "x.pkl"), est, batchsize=4, log=lambda m: None)
