"""Every person of every frame on the device (PoseEstimator.every_person, opb_pose_every_*) against the host loop it
replaces: Body, util.handDetect on every person, Hand on every box it returns (motion.pose_mats_every_person) -- bit for
bit."""
import ctypes

import numpy as np
import pytest

from oracle import openpose_oracle as O

pytestmark = pytest.mark.gpu

# Random weights usually find nobody.  These Kaiming body weights and blurred-noise frames were found once, by a search
# on the GPU over body seeds and blur widths, to make Body assemble several persons with whole arms per frame, so that
# the hand half runs on many person-derived boxes.
BODY_SEED, BODY_SCALES, BLUR, SIZE = 62, [0.5, 1.0], 2.0, (240, 320)
CHUNK = 8                                     # hand slots per chunk of the device path


def _frames(n, seed, size=SIZE, blur=BLUR):
    import cv2
    rng = np.random.default_rng(seed)
    H, W = size
    return np.stack([cv2.GaussianBlur(rng.integers(0, 256, (H, W, 3), dtype=np.uint8), (0, 0), blur) for _ in range(n)])


@pytest.fixture(scope="module")
def ests():
    from pytorch_openpose_b200 import Body, Hand
    return (Body(O.make_weights("body", BODY_SEED, "kaiming"), scale_search=BODY_SCALES),
            Hand(O.make_weights("hand", 5, "kaiming"), scale_search=[0.5, 1.0]))


@pytest.fixture(scope="module")
def est(ests):
    from pytorch_openpose_b200 import motion
    return motion.PoseEstimator(*ests)


def _host(ests, frames):
    from pytorch_openpose_b200 import motion
    return [motion.pose_mats_every_person(f, *ests) for f in frames]


def _assert_same(out, ref, what=""):
    assert len(out) == len(ref), what
    for f, (a, b) in enumerate(zip(out, ref)):
        assert a.shape == b.shape and a.dtype == np.float64, (what, f, a.shape, b.shape)
        assert np.array_equal(a, b), (what, f, np.argwhere(a != b)[:5])


def _boxes(body, frames):
    """hand boxes util.handDetect returns per frame"""
    from pytorch_openpose_b200 import util
    return [len(util.handDetect(*body(f), f)) for f in frames]


def _every_select(candidate, subset, H, W):
    from pytorch_openpose_b200 import _lib
    cand = np.ascontiguousarray(candidate, dtype=np.float64).reshape(-1, 4)
    sub = np.ascontiguousarray(subset, dtype=np.float64).reshape(-1, 20)
    records = np.full((len(sub), 60, 3), np.nan)
    boxes = np.zeros((2 * len(sub), 5), dtype=np.int32)
    _lib.check(_lib.lib().opb_pose_every_select(_lib.context(0), cand.ctypes.data, len(cand), sub.ctypes.data, len(sub),
                                                H, W, records.ctypes.data, boxes.ctypes.data))
    used = boxes[:, 4] >= 0
    assert (boxes[~used] == -1).all() and used[:used.sum()].all()     # the list is compacted
    return records, [tuple(int(v) for v in b) for b in boxes[used]]


def test_rows_and_boxes_equal_handdetect_on_random_scenes():
    """0-8 random persons (missing joints, arms leaving the frame, collapsed arms that give boxes of width 0): the
    records' body rows equal the subset / candidate copy, and the compacted box list equals util.handDetect on the whole
    subset, entry for entry, each box tagged with its person."""
    from pytorch_openpose_b200 import util
    rng = np.random.default_rng(17)
    H, W = 240, 320
    img = np.zeros((H, W, 3), np.uint8)
    empty = listed = 0
    for trial in range(300):
        n_people = int(rng.integers(0, 9))
        cand, rows = [], []
        for p in range(n_people):
            row = -np.ones(20)
            collapse = rng.random() < 0.15
            for part in range(18):
                if rng.random() < 0.8:
                    row[part] = len(cand)
                    x = float(rng.integers(0, W)) if rng.random() < 0.85 else float(W - 1)
                    y = float(rng.integers(0, H)) if rng.random() < 0.9 else float(H - 1)
                    if collapse and part in (3, 4, 6, 7) and row[part - 1] >= 0:
                        x, y = cand[int(row[part - 1])][:2]       # elbow / wrist on the previous joint
                    cand.append([x, y, float(rng.random()), float(len(cand))])
            row[18], row[19] = float(rng.random() * 10), float((row[:18] >= 0).sum())
            rows.append(row)
        candidate = np.array(cand).reshape(-1, 4)
        subset = np.array(rows).reshape(-1, 20)
        records, boxes = _every_select(candidate, subset, H, W)
        assert records.shape == (n_people, 60, 3)
        want = np.zeros((n_people, 60, 3))
        for p in range(n_people):
            for k in range(18):
                idx = int(subset[p][k])
                if idx != -1:
                    want[p, k] = candidate[idx][:3]
        assert np.array_equal(records, want), trial
        ref = util.handDetect(candidate, subset, img)
        assert [b[:4] for b in boxes] == [(x, y, w, int(l)) for x, y, w, l in ref], trial
        tagged = [(x, y, w, int(l), p) for p in range(n_people) for x, y, w, l in util.handDetect(candidate, subset[p:p + 1], img)]
        assert boxes == tagged, trial
        empty += sum(b[2] <= 0 for b in boxes)
        listed += len(boxes)
    assert empty >= 10 and listed >= 1000, (empty, listed)


def test_golden_eight_person_scene(golden):
    g = golden("body_postproc")
    records, boxes = _every_select(g["cand_p8"], g["subset_p8"], 360, 640)
    assert records.shape == (len(g["subset_p8"]), 60, 3) and not records[:, 18:].any()
    assert np.array_equal(np.array([b[:4] for b in boxes]), g["hands_p8"])


def test_records_equal_host_composition(ests, est):
    frames = _frames(6, 1)
    out = est.every_person(frames)
    ref = _host(ests, frames)
    _assert_same(out, ref)
    boxes = _boxes(ests[0], frames)
    assert sum(len(r) >= 2 and b > 0 for r, b in zip(ref, boxes)) >= 2, ([len(r) for r in ref], boxes)
    assert any((r[:, 18:, 2] > 0).any() for r in out)              # hands were really estimated
    one = est.every_person(frames[2])                              # one frame -> one array
    assert np.array_equal(one, ref[2])


def test_chunks_and_batch_size(ests, est):
    """One batch with more boxes than a chunk holds, not a multiple of it; the same frames in batches of 1 and of n."""
    pool = _frames(24, 2)
    counts = _boxes(ests[0], pool)
    n, V = 0, 0
    while n < len(pool) and (V <= CHUNK or V % CHUNK == 0):
        V += counts[n]
        n += 1
    assert V > CHUNK and V % CHUNK != 0, counts
    frames = pool[:n]
    ref = _host(ests, frames)
    whole = est.every_person(frames)
    _assert_same(whole, ref, "batch of %d, %d boxes" % (n, V))
    single = [est.every_person(f) for f in frames]
    _assert_same(single, whole, "batches of 1")


def test_replay_alternation_and_second_size(ests, est):
    """Repeated calls (the body sequence and the hand chunk replay as CUDA graphs from the third use on), calls
    alternating with submit_batch on the same session pair, and a second frame size."""
    pair = est.sessions(1)[0]
    frames = _frames(5, 3)
    ref = _host(ests, frames)
    poses = est(frames)
    for _ in range(5):
        est.submit_every_person(frames, pair)
        _assert_same(est.collect_every_person(pair), ref, "repeat")
    for _ in range(3):
        est.submit_batch(frames, pair)
        assert np.array_equal(est.collect(pair), poses)
        est.submit_every_person(frames, pair)
        _assert_same(est.collect_every_person(pair), ref, "alternating")
    other = _frames(3, 4, size=(200, 360))
    other_ref = _host(ests, other)
    for _ in range(4):
        est.submit_every_person(other, pair)
        _assert_same(est.collect_every_person(pair), other_ref, "second size")
    est.submit_every_person(frames, pair)
    _assert_same(est.collect_every_person(pair), ref, "back to the first size")


def test_inputs_on_device_and_pinned(ests, est):
    import torch
    frames = _frames(4, 5)
    ref = _host(ests, frames)
    pair = est.sessions(1)[0]
    dev = torch.from_numpy(frames).cuda()
    torch.cuda.synchronize()
    est.submit_every_person((dev.data_ptr(), frames.shape[:3]), pair, where=1)
    _assert_same(est.collect_every_person(pair), ref, "device")
    pinned = torch.from_numpy(frames).pin_memory()
    est.submit_every_person(pinned.numpy(), pair, where=2)
    _assert_same(est.collect_every_person(pair), ref, "pinned")


def test_nobody_found_launches_no_hand_work():
    from pytorch_openpose_b200 import Body, Hand, _lib, motion
    body = Body(O.make_weights("body", 0), scale_search=[0.5, 1.0])
    hand = Hand(O.make_weights("hand", 5, "kaiming"), scale_search=[0.5, 1.0])
    e = motion.PoseEstimator(body, hand)
    frames = _frames(3, 6)
    for _ in range(3):
        out = e.every_person(frames)
        assert [r.shape for r in out] == [(0, 60, 3)] * 3
        body.batch(frames)
    before = _lib.launch_count()
    body.batch(frames)
    body_only = _lib.launch_count() - before
    before = _lib.launch_count()
    out = e.every_person(frames)
    assert _lib.launch_count() - before == body_only + 1            # the body sequence and the rows-and-boxes kernel
    assert [r.shape for r in out] == [(0, 60, 3)] * 3


def test_bad_arguments(ests, est, monkeypatch):
    from pytorch_openpose_b200 import Hand, _lib
    pair = est.sessions(1)[0]
    frames = _frames(2, 7)
    with pytest.raises(_lib.OpbError):
        est.submit_every_person(np.zeros((65, 16, 16, 3), np.uint8), pair)
    with pytest.raises(_lib.OpbError):
        est.submit_every_person(frames[:0], pair)
    with pytest.raises(_lib.OpbError):
        est.submit_every_person(frames, (pair[1], pair[0]))        # session kinds swapped
    with pytest.raises(_lib.OpbError):
        est.submit_every_person(frames, (pair[0], pair[0]))        # two body sessions
    fresh = ests[0].net.session()                                  # nothing in flight on a fresh body session
    assert _lib.lib().opb_pose_every_wait(fresh.handle, (ctypes.c_int * 1)(), None) == _lib.OPB_ERR_INVALID
    with pytest.raises(ValueError):
        est.submit_every_person(frames[..., :2], pair)
    other_ctx = ctypes.c_void_p()
    _lib.check(_lib.lib().opb_context_create(0, ctypes.byref(other_ctx)))
    monkeypatch.setitem(_lib._contexts, "second", other_ctx)
    other = Hand(O.make_weights("hand", 5, "kaiming"), scale_search=[0.5, 1.0], device="second")
    with pytest.raises(_lib.OpbError):
        est.submit_every_person(frames, (pair[0], other.net.session()))   # networks on different contexts
    est.submit_every_person(frames, pair)                           # the pair still works
    _assert_same(est.collect_every_person(pair), _host(ests, frames))


def test_every_person_grows_result_buffers():
    """Frames whose peaks / limb pairs / person rows overflow the (here: tiny) initial body buffers, and more persons
    than the (here: tiny) initial records hold: the device path grows them, repeats the rows and boxes, and still equals
    the host composition -- also on the following calls (re-captured graphs)."""
    import os
    import subprocess
    import sys
    code = r'''
import numpy as np, cv2
from oracle import openpose_oracle as O
from pytorch_openpose_b200 import Body, Hand, motion
from tests import test_gpu_pose_every as T
frames = T._frames(2, 21, blur=1.5)
body = Body(O.make_weights("body", T.BODY_SEED, "kaiming"), scale_search=[1.0])
hand = Hand(O.make_weights("hand", 5, "kaiming"), scale_search=[0.5, 1.0])
est = motion.PoseEstimator(body, hand)
persons = 0
refs = [motion.pose_mats_every_person(f, body, hand) for f in frames]
c, s = body(frames[0])
assert len(c) > 64 and len(s) > 4, (len(c), len(s))    # more peaks and person rows than the tiny buffers hold
for rep in range(4):
    out = est.every_person(frames)
    for f in range(2):
        assert out[f].shape == refs[f].shape and np.array_equal(out[f], refs[f]), (rep, f)
        persons += len(refs[f])
print("EVERY-GROWTH-OK persons", persons)
'''
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, OPB_TEST_SMALL_BUFFERS="1", PYTHONPATH=root)
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True, timeout=600)
    assert "EVERY-GROWTH-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
