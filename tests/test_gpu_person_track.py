"""Person tracks on the device (opb_tracker_*, PoseEstimator.tracker, extract_every_person_from_video) against the host
rule motion.PersonLinker -- ids equal exactly, float ties included."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import openpose_oracle as O
from tests.test_gpu_pose_every import BODY_SEED, _frames, _host, _assert_same
from tests.test_person_linker import frame, person

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def crowd_sequence(seed, frames=30, max_persons=300, grid=False):
    """persons that move, appear and vanish; 0 to max_persons per frame; on an integer grid many costs tie exactly"""
    rng = np.random.default_rng(seed)
    pos = rng.uniform(0, 40 * np.sqrt(max_persons), (max_persons, 2))
    out = []
    for t in range(frames):
        pos += rng.normal(0, 3, pos.shape)
        share = 0.0 if t % 11 == 5 else rng.uniform(0.3, 1.0)
        here = np.nonzero(rng.random(max_persons) < share)[0]
        rng.shuffle(here)
        recs = []
        for p in here:
            x, y = (np.round(pos[p] / 4) * 4) if grid else pos[p]
            joints = np.nonzero(rng.random(18) < 0.75)[0]
            recs.append(person(x, y, joints=joints, score=0.1 + rng.random()))
        out.append(frame(*recs))
    return out


def host_ids(seq, max_gap, max_dist, min_joints=3):
    from pytorch_openpose_b200 import motion
    lk = motion.PersonLinker(max_gap, max_dist, min_joints)
    return [lk.link(r) for r in seq]


def device_ids(seq, max_gap, max_dist, min_joints=3, splits=(7, 1, 5)):
    """linked through opb_tracker_link_host in calls of varying frame counts (the state carries across calls)"""
    from pytorch_openpose_b200 import _lib
    tr = _lib.Tracker(_lib.context(), max_gap, max_dist, min_joints)
    out, i, s = [], 0, 0
    while i < len(seq):
        n = splits[s % len(splits)]
        out += tr.link_host(seq[i:i + n])
        i, s = i + n, s + 1
    return out, tr


def _same_ids(a, b):
    assert len(a) == len(b)
    for t, (x, y) in enumerate(zip(a, b)):
        assert np.array_equal(np.asarray(x), np.asarray(y)), (t, x, y)


@pytest.mark.parametrize("seed,max_persons,grid", [(0, 12, False), (1, 12, True), (2, 60, True), (3, 300, False),
                                                    (4, 300, True)])
def test_kernel_ids_equal_host_linker(seed, max_persons, grid):
    seq = crowd_sequence(seed, max_persons=max_persons, grid=grid)
    for max_gap, max_dist, min_joints in ((3, 12.0, 3), (1, 8.0, 5), (6, 30.0, 1)):
        ref = host_ids(seq, max_gap, max_dist, min_joints)
        dev, tr = device_ids(seq, max_gap, max_dist, min_joints)
        _same_ids(dev, ref)
        assert tr.state()[1:] == (1 + max(int(i.max()) for i in ref if len(i)), len(seq))


def test_exact_ties_on_the_device():
    seqs = [[frame(person(10, 0), person(0, 0)), frame(person(5, 0))],
            [frame(person(0, 0)), frame(person(3, 0), person(-3, 0))],
            [frame(person(0, 0)), frame(person(-3, 0), person(3, 0))]]
    for seq in seqs:
        _same_ids(device_ids(seq, 2, 10.0)[0], host_ids(seq, 2, 10.0))


def test_capacity_growth_from_tiny_buffers():
    code = r'''
import numpy as np
from tests import test_gpu_person_track as T
for seed, mp in ((5, 300), (6, 40)):
    seq = T.crowd_sequence(seed, frames=20, max_persons=mp, grid=True)
    T._same_ids(T.device_ids(seq, 4, 20.0, splits=(1, 6, 3))[0], T.host_ids(seq, 4, 20.0))
print("TRACK-GROWTH-OK")
'''
    env = dict(os.environ, OPB_TEST_SMALL_BUFFERS="1", PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert "TRACK-GROWTH-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ---- end to end on the every-person pipeline -----------------------------------------------------------------------
CLIP = 12
GATE = dict(max_gap=3, max_dist=24.0)


def shifted_clip(n=CLIP):
    """one blurred-noise frame shifted by 3 pixels per frame: the same persons recur, a little further right"""
    base = _frames(1, 7, size=(240, 400))[0]
    return np.stack([base[:, 60 - 3 * t:380 - 3 * t] for t in range(n)])


@pytest.fixture(scope="module")
def ests():
    from pytorch_openpose_b200 import Body, Hand
    return (Body(O.make_weights("body", BODY_SEED, "kaiming"), scale_search=[0.5, 1.0]),
            Hand(O.make_weights("hand", 5, "kaiming"), scale_search=[0.5, 1.0]))


@pytest.fixture(scope="module")
def est(ests):
    from pytorch_openpose_b200 import motion
    return motion.PoseEstimator(*ests)


@pytest.fixture(scope="module")
def clip_ref(ests):
    frames = shifted_clip()
    return frames, _host(ests, frames)


def linked(est, frames, batch, tracker):
    recs, ids = [], []
    for i in range(0, len(frames), batch):
        r, d = est.every_person(frames[i:i + batch], tracker)
        recs += r
        ids += d
    return recs, ids


def test_device_ids_equal_host_linker_end_to_end(est, clip_ref):
    frames, ref = clip_ref
    tr = est.tracker(**GATE)
    recs, ids = linked(est, frames, 4, tr)
    _assert_same(recs, ref, "records")
    _same_ids(ids, host_ids(ref, **GATE))
    assert sum(len(r) for r in ref) >= 2 * CLIP
    seen = {}
    for t, d in enumerate(ids):
        for i in d:
            seen.setdefault(int(i), []).append(t)
    assert max(v[-1] - v[0] + 1 for v in seen.values()) >= 0.75 * CLIP, seen    # a track spans most of the clip


def test_batch_size_does_not_change_ids(est, clip_ref):
    frames, ref = clip_ref
    want = host_ids(ref, **GATE)
    for batch in (1, 3, 8):
        tr = est.tracker(**GATE)
        _same_ids(linked(est, frames, batch, tr)[1], want)
        tr.reset()                                                                 # reset: as new
        _same_ids(linked(est, frames, batch, tr)[1], want)


def test_two_session_pairs_and_padded_batches(est, clip_ref):
    frames, ref = clip_ref
    want = host_ids(ref, **GATE)
    pairs = est.sessions(2)
    # two pairs in flight: submit two, then alternate collect / submit; collects run in submission order
    tr = est.tracker(**GATE)
    got, pending = [], []
    for k, i in enumerate(range(0, CLIP, 3)):
        if len(pending) == 2:
            got += est.collect_every_person(pending.pop(0), tracker=tr)[1]
        pair = pairs[k % 2]
        est.submit_every_person(frames[i:i + 3], pair)
        pending.append(pair)
    while pending:
        got += est.collect_every_person(pending.pop(0), tracker=tr)[1]
    _same_ids(got, want)
    # a padded last batch: 8 frames, then 4 real frames padded to 8 with n_link=4
    tr = est.tracker(**GATE)
    _, first = est.every_person(frames[:8], tr)
    padded = np.concatenate([frames[8:], np.repeat(frames[-1:], 4, axis=0)])
    est.submit_every_person(padded)
    recs, last = est.collect_every_person(tracker=tr, n_link=4)
    assert all((d == -1).all() for d in last[4:])
    _same_ids(first + last[:4], want)
    plain = est.tracker(**GATE)
    linked(est, frames, 4, plain)
    assert tr.state() == plain.state() and tr.state()[2] == CLIP


def test_bad_arguments(est, clip_ref):
    from pytorch_openpose_b200 import _lib
    frames, _ = clip_ref
    for args in ((0, 5.0, 3), (2, -1.0, 3), (2, float("nan"), 3), (2, 5.0, 0), (2, 5.0, 19)):
        with pytest.raises(_lib.OpbError):
            est.tracker(*args)
    tr = est.tracker(**GATE)
    est.submit_every_person(frames[:2])
    with pytest.raises(_lib.OpbError):
        est.collect_every_person(tracker=tr, n_link=3)
    assert tr.state() == (0, 0, 0)
    est.submit_every_person(frames[:2])
    est.collect_every_person()                                                     # untracked: no ids to fetch
    bs = est.sessions(1)[0][0]
    ids = np.empty(64, dtype=np.int32)
    assert _lib.lib().opb_pose_every_fetch_ids(bs.handle, ids.ctypes.data, 64) == _lib.OPB_ERR_INVALID
    counts = np.array([-1], dtype=np.int32)
    assert _lib.lib().opb_tracker_link_host(tr.handle, None, counts.ctypes.data, 1, None) == _lib.OPB_ERR_INVALID


# ---- the video job -------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def video(tmp_path_factory):
    import cv2
    path = str(tmp_path_factory.mktemp("vid") / "clip.avi")
    frames = shifted_clip(19)
    w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (frames.shape[2] + 20, frames.shape[1] + 10))
    assert w.isOpened()
    for f in frames:
        w.write(np.pad(f, ((5, 5), (10, 10), (0, 0))))
    w.release()
    return path


def test_job_device_path_equals_host_path(ests, video, tmp_path):
    import joblib
    from pytorch_openpose_b200 import extract as E
    body, hand = ests
    rec = [(10, 5), (330, 245)]
    host = E.extract_every_person_from_video(video, str(tmp_path / "h.pkl"), rec, lambda f: body(f), lambda c: hand(c),
                                             max_gap=3, batch=4, log=lambda s: None)
    assert host["count"] == 19 and max(len(m) for _, m in host["tracks"]) >= 10
    for workers in (1, 2):
        logs = []
        out = E.extract_every_person_from_video(video, str(tmp_path / "d.pkl"), rec, body, hand, max_gap=3, batch=4,
                                                decode_workers=workers, log=logs.append)
        saved = joblib.load(str(tmp_path / "d.pkl"))
        assert saved["count"] == out["count"] == 19 and len(saved["tracks"]) == len(host["tracks"]), workers
        for (f1, m1), (f2, m2) in zip(saved["tracks"], host["tracks"]):
            assert f1 == f2 and m1.shape == m2.shape and m1.dtype == np.float64 and np.array_equal(m1, m2), workers
        assert logs[-1].endswith("d.pkl is saved!")
