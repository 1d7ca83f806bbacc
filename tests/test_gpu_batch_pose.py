"""The one-pass body + hand job on the device (BatchPoseEstimator, opb_batch_pose_*, extract.batch_bodyhand_extraction)
against the two-pass composition it replaces: Batch_body -> extract.body_pose (Batch_body_extraction), then
Batch_hand.track on that MotionMat (Batch_hand_extraction), srcmx/Batch_motion_Estimation.py:19-112."""
import numpy as np
import pytest

from oracle import openpose_oracle as O
from pytorch_openpose_b200 import extract
from tests.test_gpu_hand_track import _cv2_optimized, _host

pytestmark = pytest.mark.gpu

# Random weights usually find nobody.  These Kaiming body weights and blurred-noise frames were found once, by a search
# on the GPU over body seeds and blur widths, to make Batch_body assemble people with whole arms (shoulder, elbow and
# wrist) on every frame at all three test sizes, so that the hand half really runs on person-derived boxes.
BODY_SEED, BLUR = 62, 1.5


def _frames(n, H, W, seed):
    import cv2
    rng = np.random.default_rng(seed)
    return np.stack([cv2.GaussianBlur(rng.integers(0, 256, (H, W, 3), dtype=np.uint8), (0, 0), BLUR) for _ in range(n)])


@pytest.fixture(scope="module")
def ests():
    from pytorch_openpose_b200 import Batch_body, Batch_hand
    return Batch_body(O.make_weights("body", BODY_SEED, "kaiming")), Batch_hand(O.make_weights("hand", 5, "kaiming"))


@pytest.fixture(scope="module")
def est(ests):
    from pytorch_openpose_b200 import BatchPoseEstimator
    return BatchPoseEstimator(*ests)


def _motion(body, frames):
    """MotionMat of Batch_body_extraction: body_pose on the fetched Batch_body results."""
    rows = []
    for lo in range(0, len(frames), 16):
        body.submit_frames(frames[lo:lo + 16])
        rows.extend(extract.body_pose(c, s)[0] for c, s in body.collect())
    return np.stack(rows)


def _two_pass(ests, frames, boxsize=368):
    body, hand = ests
    motion = _motion(body, frames)
    return motion, hand.track(frames, motion, boxsize)


def _people(motion, hands):
    """(frames with a chosen person, frames with at least one hand key point inside a box)"""
    return int(motion.any(axis=(1, 2)).sum()), int((hands[:, :, :2] != 0).any(axis=(1, 2)).sum())


def test_rows_equal_two_pass_composition(ests, est):
    chosen = with_hand = 0
    for (H, W), n, seed in (((240, 320), 40, 1), ((720, 1280), 16, 2), ((96, 72), 20, 3)):
        frames = _frames(n, H, W, seed)
        motion, hands = est(frames)
        ref_m, ref_h = _two_pass(ests, frames)
        assert motion.shape == (n, 18, 3) and hands.shape == (n, 42, 3)
        assert np.array_equal(motion, ref_m), (H, W, np.argwhere(motion != ref_m)[:5])
        assert np.array_equal(hands, ref_h), (H, W, np.argwhere(hands != ref_h)[:5])
        with _cv2_optimized(False):                              # the host hand path with OpenCV's own resize
            assert np.array_equal(hands, _host(ests[1], frames, ref_m)[0]), (H, W)
        c, h = _people(motion, hands)
        chosen += c
        with_hand += h
    assert chosen >= 40 and with_hand >= 20, (chosen, with_hand)


def test_batch_size_does_not_change_rows(est):
    frames = _frames(32, 240, 320, 7)
    rows = []
    for n in (1, 7, 32):
        est.submit(frames[32 - n:])
        m, h = est.collect()
        rows.append((m[-1], h[-1]))
    for m, h in rows[1:]:
        assert np.array_equal(m, rows[0][0]) and np.array_equal(h, rows[0][1])


def test_graph_replay_inputs_and_bad_arguments(ests):
    import torch
    from pytorch_openpose_b200 import BatchPoseEstimator, _lib
    body, hand = ests
    e = BatchPoseEstimator(body, hand)
    pair = e.sessions(1)[0]
    frames = _frames(6, 240, 320, 9)
    outs = []
    for _ in range(5):                                           # the third use on is a CUDA graph
        e.submit(frames, pair)
        outs.append(e.collect(pair))
    for m, h in outs[1:]:
        assert np.array_equal(m, outs[0][0]) and np.array_equal(h, outs[0][1])
    ref = _two_pass(ests, frames)
    assert np.array_equal(outs[0][0], ref[0]) and np.array_equal(outs[0][1], ref[1])
    # the crops of the last batch are the hand-track crops of the same frames and track
    crops = np.empty((12, 368, 368, 3), np.uint8)
    _lib.check(_lib.lib().opb_hand_track_crops(pair[1].handle, crops.ctypes.data))
    hand.submit_track(frames, ref[0])
    hand.collect_track()
    assert np.array_equal(crops, hand.track_crops())
    big = _frames(6, 480, 640, 11)                               # tables regrow, buffers move
    big_ref = _two_pass(ests, big)
    for _ in range(4):
        e.submit(big, pair)
        m, h = e.collect(pair)
        assert np.array_equal(m, big_ref[0]) and np.array_equal(h, big_ref[1])
    for _ in range(2):                                           # and back to the small frames
        e.submit(frames, pair)
        m, h = e.collect(pair)
        assert np.array_equal(m, outs[0][0]) and np.array_equal(h, outs[0][1])
    for t in (torch.from_numpy(frames).cuda(), torch.from_numpy(frames).pin_memory()):
        e.submit(t, pair)
        m, h = e.collect(pair)
        assert np.array_equal(m, outs[0][0]) and np.array_equal(h, outs[0][1])
    with pytest.raises(_lib.OpbError):
        e.submit(frames, (pair[1], pair[0]))                     # session kinds swapped
    with pytest.raises(_lib.OpbError):
        e.submit(frames, (pair[0], pair[0]))                     # two body sessions
    with pytest.raises(_lib.OpbError):
        e.submit(np.zeros((65, 16, 16, 3), np.uint8), pair)
    with pytest.raises(_lib.OpbError):
        e.submit(frames[:0], pair)
    with pytest.raises(_lib.OpbError):
        e.submit(frames, pair, boxsize=100)
    with pytest.raises(ValueError):
        e.submit(frames[..., :2], pair)
    with pytest.raises(ValueError):
        e.submit(frames[0], pair)
    e.submit(frames, pair)
    m, h = e.collect(pair)
    assert np.array_equal(m, outs[0][0]) and np.array_equal(h, outs[0][1])


def test_batch_pose_grows_result_buffers():
    """Frames whose peaks / limb pairs / person rows overflow the (here: tiny) initial buffers: the one-pass job grows
    them, repeats the body post-processing of those frames and the hand half of the batch, and still equals the two-pass
    composition -- on the first call after a graph was captured on light frames, and on the re-captured graph."""
    import os
    import subprocess
    import sys
    code = r'''
import numpy as np
from oracle import openpose_oracle as O
from pytorch_openpose_b200 import Batch_body, Batch_hand, BatchPoseEstimator
from tests import test_gpu_batch_pose as T
body = Batch_body(O.make_weights("body", T.BODY_SEED, "kaiming"))
hand = Batch_hand(O.make_weights("hand", 5, "kaiming"))
e = BatchPoseEstimator(body, hand)
light = np.full((3, 720, 1280, 3), 128, np.uint8)
for _ in range(3):                                  # graph captured on frames that fit the buffers
    e(light)
heavy = T._frames(3, 720, 1280, 21)
most = [0, 0]
for rep in range(3):
    m, h = e(heavy)
    ref = T._two_pass((body, hand), heavy)
    assert np.array_equal(m, ref[0]) and np.array_equal(h, ref[1]), rep
body.submit_frames(heavy)
for c, s in body.collect():
    most = [max(most[0], len(c)), max(most[1], len(s))]
assert most[0] > 64 and most[1] > 4, most          # more peaks and person rows than the tiny buffers hold
print("BATCH-POSE-GROWTH-OK", most, T._people(m, h))
'''
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, OPB_TEST_SMALL_BUFFERS="1", PYTHONPATH=root)
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True, timeout=600)
    assert "BATCH-POSE-GROWTH-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def _video(path, n, w, h):
    import cv2
    wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (w, h))
    assert wr.isOpened()
    rng = np.random.default_rng(31)
    for _ in range(n):
        wr.write(cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), BLUR))
    wr.release()


@pytest.mark.parametrize("workers", [1, 2])
def test_video_job_equals_two_jobs(tmp_path, ests, workers):
    import joblib
    body, hand = ests
    path = str(tmp_path / "v.avi")
    _video(path, 11, 320, 240)
    rec = [(16, 8), (304, 232)]
    one, two = [], []
    m, h = extract.batch_bodyhand_extraction(path, str(tmp_path / "b1.pkl"), str(tmp_path / "h1.pkl"), 4, rec, body, hand,
                                             log=one.append, decode_workers=workers, sessions=2)
    m2 = extract.batch_body_extraction(path, str(tmp_path / "b2.pkl"), 4, rec, body, log=two.append,
                                       decode_workers=workers)
    h2 = extract.batch_hand_extraction(path, m2, rec, str(tmp_path / "h2.pkl"), hand, batchsize=4, log=two.append,
                                       decode_workers=workers)
    assert m.shape == (11, 18, 3) and h.shape == (11, 42, 3) and m.dtype == h.dtype == np.float64
    for a, b in (("b1.pkl", "b2.pkl"), ("h1.pkl", "h2.pkl")):
        fa, fb = joblib.load(str(tmp_path / a)), joblib.load(str(tmp_path / b))
        assert fa.shape == fb.shape and fa.dtype == fb.dtype and np.array_equal(fa, fb), a
    assert np.array_equal(m, m2) and np.array_equal(h, h2)
    assert sorted(l.replace("1.pkl", "2.pkl") for l in one) == sorted(two)
    assert (m[:, :, 2] > 0).any()                                # people were found in the decoded frames
