"""CUDA graph keys of the sessions: a job replays its captured launch sequence only while nothing it reads has moved.
Every check compares against the eager result of the same inputs on the same session pair (profiling runs every job
eagerly), bit for bit, and counts captures and replays with opb_session_graph_stats."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import openpose_oracle as O
from tests.test_gpu_pose_every import BODY_SEED, _frames

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOX = 184                                     # Batch_hand boxsize of the batched jobs


class Models(object):
    def __init__(self, body_scales=(0.5, 1.0)):
        from pytorch_openpose_b200 import Batch_body, Batch_hand, Body, BatchPoseEstimator, Hand, motion
        wb, wh = O.make_weights("body", BODY_SEED, "kaiming"), O.make_weights("hand", 5, "kaiming")
        self.body, self.hand = Body(wb, scale_search=list(body_scales)), Hand(wh, scale_search=[0.5, 1.0])
        self.bb, self.bh = Batch_body(wb), Batch_hand(wh)
        self.est, self.best = motion.PoseEstimator(self.body, self.hand), BatchPoseEstimator(self.bb, self.bh)

    def pair(self):
        return self.body.net.session(), self.hand.net.session()

    def jobs(self, pair, frames, poses=None):
        """name -> (session whose graphs run the job, one call: submit + collect)"""
        bs, hs = pair
        m = self
        crops = np.stack(_crops([96] * 4, 1))
        crop_list = _crops([40, 77, 120, 96, 150], 2)
        poses = np.zeros((len(frames), 18, 3)) if poses is None else poses

        def call(submit, collect):
            submit()
            return collect()
        return {
            "Body": (bs, lambda: call(lambda: m.body.submit_batch(frames, session=bs), lambda: m.body.collect_batch(bs))),
            "Batch_body": (bs, lambda: call(lambda: m.bb.submit_frames(frames, session=bs), lambda: m.bb.collect(bs))),
            "Pose": (bs, lambda: call(lambda: m.est.submit_batch(frames, pair=pair), lambda: m.est.collect(pair))),
            "Every": (bs, lambda: call(lambda: m.est.submit_every_person(frames, pair=pair),
                                       lambda: m.est.collect_every_person(pair))),
            "BatchPose": (bs, lambda: call(lambda: m.best.submit(frames, pair=pair, boxsize=BOX),
                                           lambda: m.best.collect(pair))),
            "BatchEvery": (bs, lambda: call(lambda: m.best.submit_every_person(frames, pair=pair, boxsize=BOX),
                                            lambda: m.best.collect_every_person(pair))),
            "Hand": (hs, lambda: call(lambda: m.hand.submit(crops, session=hs), lambda: m.hand.collect(hs))),
            "Crops": (hs, lambda: call(lambda: m.hand.submit(crop_list, session=hs), lambda: m.hand.collect(hs))),
            "HandTrack": (hs, lambda: call(lambda: m.bh.submit_track(frames, poses, session=hs, boxsize=BOX),
                                           lambda: m.bh.collect_track(hs))),
        }


def _crops(sides, seed):
    import cv2
    rng = np.random.default_rng(seed)
    return [cv2.GaussianBlur(rng.integers(0, 256, (w, w, 3), dtype=np.uint8), (0, 0), 2) for w in sides]


def _stats(session):
    from pytorch_openpose_b200 import _lib
    c, r = ctypes.c_longlong(), ctypes.c_longlong()
    _lib.check(_lib.lib().opb_session_graph_stats(session.handle, ctypes.byref(c), ctypes.byref(r)))
    return c.value, r.value


def _eager(session, run):
    session.set_profiling(True)
    try:
        return run()
    finally:
        session.set_profiling(False)


def _same(a, b):
    if isinstance(a, (list, tuple)):
        return isinstance(b, (list, tuple)) and len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b)


def _counted(session, run, want, what):
    """one call: its result equals `want`; returns (captures, replays) of the call"""
    c0, r0 = _stats(session)
    assert _same(run(), want), what
    c1, r1 = _stats(session)
    return c1 - c0, r1 - r0


def recaptures_once(session, run, grow, what):
    """`run` replays a captured graph; after `grow` its next call re-captures its graphs, once, and the calls after that
    replay again -- all equal to the eager result."""
    want = _eager(session, run)
    for _ in range(3):                        # two eager uses, then the capture
        assert _same(run(), want), what
    captures, graphs = _counted(session, run, want, what)
    assert captures == 0 and graphs >= 1, (what, captures, graphs)
    grow()
    captures, replays = _counted(session, run, want, what + " after the growth")
    assert captures >= 1 and captures + replays == graphs, (what, captures, replays, graphs)
    for _ in range(2):
        assert _counted(session, run, want, what + " later") == (0, graphs), what


@pytest.fixture(scope="module")
def m():
    return Models()


@pytest.fixture(scope="module")
def frames():
    return _frames(2, 31)


@pytest.fixture(scope="module")
def poses(m, frames):
    return m.best(frames, boxsize=BOX)[0]


def test_pose_after_the_pose_buffers_grew_under_a_captured_graph(m):
    """every_person sizes everything but the pose buffers; three calls on 2 frames capture the Pose graph with pose
    buffers of 2 frames; 4 frames grow them (nothing else grows); 2 frames again must not replay over the freed ones."""
    from pytorch_openpose_b200 import motion
    est = motion.PoseEstimator(m.body, m.hand)
    four = _frames(4, 32, size=(720, 1280))
    est.every_person(four)
    first = [est(four[:2]) for _ in range(3)]
    est(four)
    again = est(four[:2])
    bs, _ = est.sessions(1)[0]
    want = _eager(bs, lambda: est(four[:2]))
    assert all(_same(f, want) for f in first)
    assert _same(again, want)


def test_alternating_jobs_replay_without_capturing(m, frames, poses):
    pair = m.pair()
    jobs = m.jobs(pair, frames, poses)
    want = {k: _eager(s, run) for k, (s, run) in jobs.items()}
    assert sum(len(r) for r in want["Every"]) > 0, "no person found: the hand chunks would not run"
    for _ in range(3):                        # two eager uses of every job, then the captures
        for k, (s, run) in jobs.items():
            assert _same(run(), want[k]), k
    before = [_stats(s) for s in pair]
    for rnd in range(10):
        for k, (s, run) in jobs.items():
            assert _same(run(), want[k]), (rnd, k)
    after = [_stats(s) for s in pair]
    assert [c for c, _ in after] == [c for c, _ in before], (before, after)
    assert after[0][1] - before[0][1] >= 10 * 6 and after[1][1] - before[1][1] == 10 * 3, (before, after)


def test_more_frames(m, frames):
    pair = m.pair()
    s, run = m.jobs(pair, frames)["Pose"]
    four = _frames(4, 33)
    recaptures_once(s, run, lambda: (m.body.submit_batch(four, session=pair[0]), m.body.collect_batch(pair[0])), "Pose")


def test_larger_frame(m, frames):
    pair = m.pair()
    s, run = m.jobs(pair, frames)["Body"]
    big = _frames(1, 34, size=(480, 640))
    recaptures_once(s, run, lambda: (m.body.submit_batch(big, session=pair[0]), m.body.collect_batch(pair[0])), "Body")


def test_other_boxsize(m, frames, poses):
    pair = m.pair()
    s, run = m.jobs(pair, frames, poses)["HandTrack"]
    recaptures_once(s, run, lambda: (m.best.submit(frames, pair=pair, boxsize=BOX + 64), m.best.collect(pair)),
                    "HandTrack")


def test_other_hand_scales(m, frames):
    from pytorch_openpose_b200 import Hand, motion
    pair = m.pair()
    s, run = m.jobs(pair, frames)["Pose"]
    other = motion.PoseEstimator(m.body, Hand(O.make_weights("hand", 5, "kaiming"), scale_search=[1.0]))
    recaptures_once(s, run, lambda: (other.submit_batch(frames, pair=pair), other.collect(pair)), "Pose")


def test_hand_net_plan_eviction(m, frames):
    pair = m.pair()
    jobs = m.jobs(pair, frames)

    def evict():                              # 7 crop counts: more CNN plans than a session keeps
        for k in range(9, 16):
            m.hand.submit(np.stack(_crops([64] * k, k)), session=pair[1])
            m.hand.collect(pair[1])
    for name in ("Pose", "Every"):
        s, run = jobs[name]
        recaptures_once(s, run, evict, name)


def test_result_and_record_growth():
    """Body results that overflow their buffers, and more persons than the every-person records hold, starting from
    tiny buffers (OPB_TEST_SMALL_BUFFERS, own process)."""
    code = r'''
import numpy as np
from tests import test_gpu_graph_keys as T
from tests.test_gpu_pose_every import _frames
m = T.Models(body_scales=[1.0])
calm, busy = _frames(2, 41, blur=6.0), _frames(2, 21, blur=1.5)

pair = m.pair()
s, run = m.jobs(pair, calm)["Body"]
def overflow():
    m.body.submit_batch(busy, session=pair[0])
    out = m.body.collect_batch(pair[0])
    assert all(len(c) > 64 and len(sub) > 4 for c, sub in out), [(len(c), len(sub)) for c, sub in out]
T.recaptures_once(s, run, overflow, "Body")

pair = m.pair()
jobs = m.jobs(pair, calm)
s, run = jobs["Every"]
m.body.submit_batch(busy, session=pair[0])          # the body buffers of the plan fit the busy frames from here on
m.body.collect_batch(pair[0])
few = sum(len(r) for r in run())
cap = 2
while cap < few:
    cap *= 2
def more_persons():
    many = sum(len(r) for r in m.jobs(pair, busy)["Every"][1]())
    assert many > cap, (few, many)
T.recaptures_once(s, run, more_persons, "Every")
print("GRAPH-GROWTH-OK")
'''
    env = dict(os.environ, OPB_TEST_SMALL_BUFFERS="1", PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert "GRAPH-GROWTH-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_waits_refuse_another_batch(m, frames, poses):
    """A wait returns the results of the last batch of its kind only while no other batch ran on the session since."""
    from pytorch_openpose_b200 import _lib
    L = _lib.lib()
    pair = bs, hs = m.pair()
    status = (ctypes.c_int * len(frames))()
    persons = (ctypes.c_int * len(frames))()
    out = np.empty((len(frames), 60, 3))
    hands = np.empty((len(frames), 42, 3))
    body_only = (lambda: (m.body.submit_batch(frames, session=bs), m.body.collect_batch(bs)),
                 lambda: (m.bb.submit_frames(frames, session=bs), m.bb.collect(bs)))
    for later in body_only:
        m.est.submit_batch(frames, pair=pair)
        m.est.collect(pair)
        later()
        assert L.opb_pose_wait(bs.handle, out.ctypes.data, status) == _lib.OPB_ERR_INVALID
        m.best.submit(frames, pair=pair, boxsize=BOX)
        m.best.collect(pair)
        later()
        assert L.opb_batch_pose_wait(bs.handle, out.ctypes.data, hands.ctypes.data, status) == _lib.OPB_ERR_INVALID
        for submit in (lambda: m.est.submit_every_person(frames, pair=pair),
                       lambda: m.best.submit_every_person(frames, pair=pair, boxsize=BOX)):
            submit()
            later()
            assert L.opb_pose_every_wait(bs.handle, persons, status) == _lib.OPB_ERR_INVALID
            tracker = m.est.tracker(1, 100.0)
            assert L.opb_pose_every_wait_tracked(bs.handle, tracker.handle, len(frames), persons,
                                                 status) == _lib.OPB_ERR_INVALID
    peaks = np.empty((8, 21, 3))
    m.bh.submit_track(frames, poses, session=hs, boxsize=BOX)
    m.bh.collect_track(hs)
    assert L.opb_hand_wait(hs.handle, peaks.ctypes.data) == _lib.OPB_ERR_INVALID
    for name in ("Pose", "BatchPose", "Every", "BatchEvery"):
        m.jobs(pair, frames)[name][1]()
        assert L.opb_hand_wait(hs.handle, peaks.ctypes.data) == _lib.OPB_ERR_INVALID, name
    m.hand.submit(np.stack(_crops([64] * 2, 3)), session=hs)
    m.hand.collect(hs)                        # a hand batch of its own is collected as before
