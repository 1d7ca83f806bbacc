"""Every person on the batched estimators on the device (BatchPoseEstimator.every_person, opb_batch_pose_every_*,
extract.batch_every_person_extraction) against the host composition that states the contract,
extract.batch_pose_mats_every_person -- bit for bit."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import openpose_oracle as O
from pytorch_openpose_b200 import extract, motion
from tests.test_gpu_batch_pose import BODY_SEED, _frames
from tests.test_gpu_hand_track import _cv2_optimized
from tests.test_gpu_person_track import _same_ids, host_ids

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 32                                    # Batch_hand crops per chunk of the device path


@pytest.fixture(scope="module")
def ests():
    from pytorch_openpose_b200 import Batch_body, Batch_hand
    return Batch_body(O.make_weights("body", BODY_SEED, "kaiming")), Batch_hand(O.make_weights("hand", 5, "kaiming"))


@pytest.fixture(scope="module")
def est(ests):
    from pytorch_openpose_b200 import BatchPoseEstimator
    return BatchPoseEstimator(*ests)


def _host(ests, frames):
    with _cv2_optimized(False):                                  # the device implements OpenCV's own resize arithmetic
        return extract.batch_pose_mats_every_person(frames, *ests)


def _assert_same(out, ref, what=""):
    assert len(out) == len(ref), what
    for f, (a, b) in enumerate(zip(out, ref)):
        assert a.shape == b.shape and a.dtype == np.float64, (what, f, a.shape, b.shape)
        assert np.array_equal(a, b), (what, f, np.argwhere(a != b)[:5])


def _with_hands(records):
    """records whose hand key points have a coordinate inside a box"""
    return sum(int((r[:, 18:, :2] != 0).any(axis=(1, 2)).sum()) for r in records)


# ---- rows and slots on given body results ---------------------------------------------------------------------------
def _batch_select(candidate, subset, H, W):
    from pytorch_openpose_b200 import _lib
    cand = np.ascontiguousarray(candidate, dtype=np.float64).reshape(-1, 4)
    sub = np.ascontiguousarray(subset, dtype=np.float64).reshape(-1, 20)
    records = np.full((len(sub), 60, 3), np.nan)
    slots = np.zeros((2 * len(sub), 6), dtype=np.int32)
    _lib.check(_lib.lib().opb_batch_pose_every_select(_lib.context(0), cand.ctypes.data, len(cand), sub.ctypes.data,
                                                      len(sub), H, W, records.ctypes.data, slots.ctypes.data))
    return records, [tuple(int(v) for v in s) for s in slots]


def _scene(rng, n_people, H, W):
    """random persons: missing joints, arms leaving the frame, collapsed arms that give boxes of width 0"""
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
                    x, y = cand[int(row[part - 1])][:2]               # elbow / wrist on the previous joint
                cand.append([x, y, float(rng.random()), float(len(cand))])
        row[18], row[19] = float(rng.random() * 10), float((row[:18] >= 0).sum())
        rows.append(row)
    return np.array(cand).reshape(-1, 4), np.array(rows).reshape(-1, 20)


def test_rows_and_slots_on_random_scenes():
    """The body rows of every subset row, and both slots of every person -- left then right, person after person --
    with the boxes of hand_crops_from_pose on exactly those rows (extract.pose_person + util.handDetect).  A hand with a
    missing joint is the invalid slot (0, 0, 0); a box of width <= 0 keeps its x, y, w and is invalid."""
    from pytorch_openpose_b200 import util
    rng = np.random.default_rng(23)
    H, W = 240, 320
    img = np.zeros((H, W, 3), np.uint8)
    empty = invalid = valid = 0
    for trial in range(300):
        n_people = int(rng.integers(0, 301)) if trial % 10 == 0 else int(rng.integers(0, 9))
        candidate, subset = _scene(rng, n_people, H, W)
        records, slots = _batch_select(candidate, subset, H, W)
        assert records.shape == (n_people, 60, 3) and len(slots) == 2 * n_people
        want = []
        for p in range(n_people):
            body = np.zeros((18, 3))
            for k in range(18):
                if int(subset[p][k]) != -1:
                    body[k] = candidate[int(subset[p][k])][:3]
            assert np.array_equal(records[p, :18], body) and not records[p, 18:].any(), (trial, p)
            found = {bool(l): (x, y, w) for x, y, w, l in util.handDetect(*extract.pose_person(body), img)}
            for left in (True, False):
                x, y, w = found.get(left, (0, 0, 0))
                want.append((x, y, w, int(w > 0), int(left), p))
                empty += left in found and w <= 0
        assert slots == want, trial
        valid += sum(s[3] for s in slots)
        invalid += sum(1 - s[3] for s in slots)
    assert empty >= 10 and valid >= 1000 and invalid >= 1000, (empty, valid, invalid)


# ---- end to end ---------------------------------------------------------------------------------------------------------
def test_records_equal_host_composition(ests, est):
    several = with_hands = 0
    big_batch = False
    for (H, W), n, seed in (((240, 320), 24, 1), ((720, 1280), 8, 2), ((96, 72), 12, 3)):
        frames = _frames(n, H, W, seed)
        out = est.every_person(frames)
        ref = _host(ests, frames)
        _assert_same(out, ref, (H, W))
        several += sum(len(r) >= 2 for r in ref)
        with_hands += _with_hands(ref)
        big_batch |= 2 * sum(len(r) for r in ref) > CHUNK
    assert several >= 4 and with_hands >= 4 and big_batch, (several, with_hands, big_batch)
    one = est.every_person(frames[2])                              # one frame -> one array
    assert np.array_equal(one, ref[2])


def test_selected_person_equals_the_one_person_path(ests, est):
    body = ests[0]
    frames = _frames(16, 240, 320, 4)
    out = est.every_person(frames)
    m, h = est(frames)
    body.submit_frames(frames)
    checked = 0
    for f, (candidate, subset) in enumerate(body.collect()):
        p = motion.select_person(candidate, subset)
        assert len(out[f]) == len(subset)
        if p is None:
            assert not m[f].any()
            continue
        assert np.array_equal(out[f][p], np.concatenate([m[f], h[f]])), f
        checked += 1
    assert checked >= 8


def test_batch_size_does_not_change_records(est):
    frames = _frames(32, 240, 320, 7)
    last = [est.every_person(frames[32 - n:])[-1] for n in (1, 7, 32)]
    for r in last[1:]:
        assert np.array_equal(r, last[0])


def test_replay_alternation_sizes_and_inputs(ests, est):
    """Repeated calls (CUDA graphs from the third use on), calls alternating with the one-person submit on the same
    session pair, a larger second frame size (tables regrow, buffers move) and back, CUDA-tensor and pinned input."""
    import torch
    pair = est.sessions(1)[0]
    frames = _frames(6, 240, 320, 9)
    ref = _host(ests, frames)
    for _ in range(5):
        est.submit_every_person(frames, pair)
        _assert_same(est.collect_every_person(pair), ref, "repeat")
    one = est(frames)
    for _ in range(3):
        est.submit(frames, pair)
        m, h = est.collect(pair)
        assert np.array_equal(m, one[0]) and np.array_equal(h, one[1])
        est.submit_every_person(frames, pair)
        _assert_same(est.collect_every_person(pair), ref, "alternating")
    big = _frames(4, 480, 640, 11)
    big_ref = _host(ests, big)
    for _ in range(4):
        est.submit_every_person(big, pair)
        _assert_same(est.collect_every_person(pair), big_ref, "second size")
    est.submit_every_person(frames, pair)
    _assert_same(est.collect_every_person(pair), ref, "back to the first size")
    for t in (torch.from_numpy(frames).cuda(), torch.from_numpy(frames).pin_memory()):
        est.submit_every_person(t, pair)
        _assert_same(est.collect_every_person(pair), ref, str(t.device))


def test_bad_arguments(ests, est):
    from pytorch_openpose_b200 import _lib
    pair = est.sessions(1)[0]
    frames = _frames(2, 64, 80, 12)
    with pytest.raises(_lib.OpbError):
        est.submit_every_person(frames, pair, boxsize=100)
    with pytest.raises(_lib.OpbError):
        est.submit_every_person(np.zeros((65, 16, 16, 3), np.uint8), pair)
    with pytest.raises(_lib.OpbError):
        est.submit_every_person(frames[:0], pair)
    with pytest.raises(_lib.OpbError):
        est.submit_every_person(frames, (pair[1], pair[0]))          # session kinds swapped
    with pytest.raises(ValueError):
        est.submit_every_person(frames[..., :2], pair)
    fresh = ests[0].net.session()                                    # nothing in flight on a fresh body session
    assert _lib.lib().opb_pose_every_wait(fresh.handle, (ctypes.c_int * 1)(), None) == _lib.OPB_ERR_INVALID
    est.submit(frames, pair)                                         # a one-person batch is not an every-person batch
    assert _lib.lib().opb_pose_every_wait(pair[0].handle, (ctypes.c_int * 2)(), None) == _lib.OPB_ERR_INVALID
    est.collect(pair)
    est.submit_every_person(frames, pair)
    with pytest.raises(_lib.OpbError):
        est.collect(pair)                                            # ... and the other way round
    _assert_same(est.collect_every_person(pair), _host(ests, frames))


def test_nobody_found_launches_no_hand_work():
    from pytorch_openpose_b200 import Batch_body, Batch_hand, BatchPoseEstimator, _lib
    body = Batch_body(O.make_weights("body", 0))
    e = BatchPoseEstimator(body, Batch_hand(O.make_weights("hand", 5, "kaiming")))
    frames = _frames(3, 240, 320, 6)
    for _ in range(3):
        assert [r.shape for r in e.every_person(frames)] == [(0, 60, 3)] * 3
        body.submit_frames(frames)
        body.collect()
    before = _lib.launch_count()
    body.submit_frames(frames)
    body.collect()
    body_only = _lib.launch_count() - before
    before = _lib.launch_count()
    out = e.every_person(frames)
    assert _lib.launch_count() - before == body_only + 1             # the body sequence and the rows-and-slots kernel
    assert [r.shape for r in out] == [(0, 60, 3)] * 3


def test_records_grow_from_tiny_buffers():
    """More persons than the (here: tiny) initial records hold, and frames that overflow the tiny body buffers: the
    device path grows them, repeats the rows and slots, and still equals the host composition -- also on the following
    calls (re-captured graphs)."""
    code = r'''
import numpy as np
from oracle import openpose_oracle as O
from pytorch_openpose_b200 import Batch_body, Batch_hand, BatchPoseEstimator
from tests import test_gpu_batch_pose_every as T
body = Batch_body(O.make_weights("body", T.BODY_SEED, "kaiming"))
hand = Batch_hand(O.make_weights("hand", 5, "kaiming"))
est = BatchPoseEstimator(body, hand)
frames = T._frames(3, 720, 1280, 21)
ref = T._host((body, hand), frames)
assert sum(len(r) for r in ref) > 8, [len(r) for r in ref]
for rep in range(4):
    T._assert_same(est.every_person(frames), ref, rep)
print("BATCH-EVERY-GROWTH-OK", [len(r) for r in ref])
'''
    env = dict(os.environ, OPB_TEST_SMALL_BUFFERS="1", PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert "BATCH-EVERY-GROWTH-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ---- tracks -----------------------------------------------------------------------------------------------------------
CLIP = 12
GATE = dict(max_gap=3, max_dist=24.0)


def shifted_clip(n=CLIP):
    """one blurred-noise frame shifted by 3 pixels per frame: the same persons recur, a little further right"""
    base = _frames(1, 240, 400, 8)[0]
    return np.stack([base[:, 60 - 3 * t:380 - 3 * t] for t in range(n)])


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


def test_device_ids_equal_host_linker(est, clip_ref):
    frames, ref = clip_ref
    tr = est.tracker(**GATE)
    recs, ids = linked(est, frames, 5, tr)
    _assert_same(recs, ref, "records")
    _same_ids(ids, host_ids(ref, **GATE))
    assert sum(len(r) for r in ref) >= 2 * CLIP
    seen = {}
    for t, d in enumerate(ids):
        for i in d:
            seen.setdefault(int(i), []).append(t)
    assert max(v[-1] - v[0] + 1 for v in seen.values()) >= 0.75 * CLIP, seen    # a track spans most of the clip


def test_two_session_pairs_padded_batch_and_failed_wait(est, clip_ref):
    from pytorch_openpose_b200 import _lib
    frames, ref = clip_ref
    want = host_ids(ref, **GATE)
    pairs = est.sessions(2)
    tr = est.tracker(**GATE)
    got, pending = [], []
    for k, i in enumerate(range(0, CLIP, 3)):
        if len(pending) == 2:
            got += est.collect_every_person(pending.pop(0), tracker=tr)[1]
        est.submit_every_person(frames[i:i + 3], pairs[k % 2])
        pending.append(pairs[k % 2])
    while pending:
        got += est.collect_every_person(pending.pop(0), tracker=tr)[1]
    _same_ids(got, want)
    # a padded last batch: 8 frames, then 4 real frames padded to 8 with n_link=4
    tr = est.tracker(**GATE)
    _, first = est.every_person(frames[:8], tr)
    padded = np.concatenate([frames[8:], np.repeat(frames[-1:], 4, axis=0)])
    est.submit_every_person(padded)
    _, last = est.collect_every_person(tracker=tr, n_link=4)
    assert all((d == -1).all() for d in last[4:])
    _same_ids(first + last[:4], want)
    assert tr.state()[2] == CLIP
    # a wait that fails links nothing
    state = tr.state()
    est.submit_every_person(frames[:2])
    with pytest.raises(_lib.OpbError):
        est.collect_every_person(tracker=tr, n_link=3)
    assert tr.state() == state


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


def test_job_device_file_equals_host_fallback_file(ests, video, tmp_path):
    import joblib
    body, hand = ests
    rec = [(10, 5), (330, 245)]
    with _cv2_optimized(False):
        host = extract.batch_every_person_extraction(video, str(tmp_path / "h.pkl"), 4, rec, lambda b: body(b),
                                                     lambda c: hand(c), max_gap=3, log=lambda s: None)
    assert host["count"] == 19 and max(len(m) for _, m in host["tracks"]) >= 10
    for workers in (1, 2):
        logs = []
        out = extract.batch_every_person_extraction(video, str(tmp_path / "d.pkl"), 4, rec, body, hand, max_gap=3,
                                                    decode_workers=workers, log=logs.append)
        saved = joblib.load(str(tmp_path / "d.pkl"))
        assert saved["count"] == out["count"] == 19 and len(saved["tracks"]) == len(host["tracks"]), workers
        for (f1, m1), (f2, m2) in zip(saved["tracks"], host["tracks"]):
            assert f1 == f2 and m1.shape == m2.shape and m1.dtype == np.float64 and np.array_equal(m1, m2), workers
        assert logs == ["d.pkl-0/19", "%s is saved!" % (tmp_path / "d.pkl")]
