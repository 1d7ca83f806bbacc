"""motion.PersonLinker (the linking rule the device tracker is held to) on hand-built sequences, a randomized property
check, and the every-person video job with estimators other than this package's (host path)."""
import numpy as np
import pytest

from pytorch_openpose_b200 import extract as E
from pytorch_openpose_b200 import motion
from tests.test_extract import REC, fake_body, fake_hand


def person(x, y, joints=range(18), score=0.5):
    """one (60, 3) record: joint j at (x + j, y + 2 j) for the given joints, the rest missing"""
    r = np.zeros((60, 3))
    for j in joints:
        r[j] = (x + j, y + 2 * j, score)
    return r


def frame(*records):
    return np.array(records).reshape(-1, 60, 3)


def test_two_persons_crossing_keep_their_ids():
    lk = motion.PersonLinker(max_gap=3, max_dist=20)
    seen = []
    for t in range(12):
        a, b = person(10 + 5 * t, 50), person(65 - 5 * t, 56)
        seen.append(list(lk.link(frame(a, b) if t % 2 else frame(b, a))))    # subset order changes from frame to frame
    assert seen == [[1, 0] if t % 2 else [0, 1] for t in range(12)]


def test_returning_within_max_gap_keeps_the_id():
    # "live for frame t when t - last <= max_gap": back max_gap frames after the last match keeps the id (max_gap - 1
    # frames without the person in between); one frame later it is a new track
    for gap, expect in ((4, 0), (5, 1)):
        lk = motion.PersonLinker(max_gap=4, max_dist=10)
        assert list(lk.link(frame(person(0, 0)))) == [0]
        for _ in range(gap - 1):
            assert list(lk.link(frame())) == []                               # frames with nobody count
        assert list(lk.link(frame(person(1, 1)))) == [expect]


def test_tracks_not_live_are_dropped_for_good():
    lk = motion.PersonLinker(max_gap=1, max_dist=10)
    lk.link(frame(person(0, 0)))
    lk.link(frame())
    lk.link(frame())
    assert list(lk.link(frame(person(0, 0), person(100, 100)))) == [1, 2]   # id 0 is not reused


def test_min_joints():
    for min_joints, expect in ((3, 1), (2, 0)):
        lk = motion.PersonLinker(max_gap=2, max_dist=10, min_joints=min_joints)
        lk.link(frame(person(0, 0, joints=[0, 1, 2, 3])))
        assert list(lk.link(frame(person(0, 0, joints=[2, 3, 4, 5])))) == [expect]     # two joints in common


def test_exact_ties_break_on_track_id_then_person_index():
    lk = motion.PersonLinker(max_gap=2, max_dist=10)
    assert list(lk.link(frame(person(10, 0), person(0, 0)))) == [0, 1]
    assert list(lk.link(frame(person(5, 0)))) == [0]                        # cost 5 to both tracks: the lower id wins
    lk = motion.PersonLinker(max_gap=2, max_dist=10)
    lk.link(frame(person(0, 0)))
    assert list(lk.link(frame(person(3, 0), person(-3, 0)))) == [0, 1]       # cost 3 from both persons: index 0 wins
    lk = motion.PersonLinker(max_gap=2, max_dist=10)
    lk.link(frame(person(0, 0)))
    assert list(lk.link(frame(person(-3, 0), person(3, 0)))) == [0, 1]


def test_cost_gate_and_absent_joints():
    lk = motion.PersonLinker(max_gap=2, max_dist=5)
    lk.link(frame(person(0, 0)))
    assert list(lk.link(frame(person(5, 0)))) == [0]                         # cost == max_dist is eligible
    assert list(lk.link(frame(person(10.5, 0)))) == [1]
    lk = motion.PersonLinker(max_gap=2, max_dist=5)
    lk.link(frame(person(0, 0, joints=range(6))))
    far = person(0, 0, joints=range(4))
    far[4:6] = [(90, 90, 0.0), (90, 90, 0.0)]                               # score 0: absent, coordinates ignored
    assert list(lk.link(frame(far))) == [0]


def test_cost_is_the_documented_float64_expression():
    lk = motion.PersonLinker(max_gap=1, max_dist=1e9)
    rng = np.random.default_rng(0)
    a, b = rng.normal(size=(60, 3)) * 100, rng.normal(size=(60, 3)) * 100
    a[:, 2], b[:, 2] = np.abs(a[:, 2]), np.abs(b[:, 2])
    lk.link(frame(a))
    lk.link(frame(b))
    s = 0.0
    for j in range(18):
        dx, dy = b[j, 0] - a[j, 0], b[j, 1] - a[j, 1]
        s = s + float(np.sqrt(dx * dx + dy * dy))
    cost = s / 18
    for gate, expect in ((cost, 0), (np.nextafter(cost, 0), 1)):
        lk = motion.PersonLinker(max_gap=1, max_dist=gate)
        lk.link(frame(a))
        assert list(lk.link(frame(b))) == [expect]


def random_sequence(seed, frames=40, max_persons=12):
    """persons that move, appear and vanish, with partial joints"""
    rng = np.random.default_rng(seed)
    pos = rng.uniform(0, 200, (max_persons, 2))
    out = []
    for _ in range(frames):
        pos += rng.normal(0, 4, pos.shape)
        here = np.nonzero(rng.random(max_persons) < 0.7)[0]
        rng.shuffle(here)
        recs = []
        for p in here:
            joints = np.nonzero(rng.random(18) < 0.7)[0]
            recs.append(person(pos[p, 0], pos[p, 1], joints=joints, score=0.1 + rng.random()))
        out.append(frame(*recs))
    return out


@pytest.mark.parametrize("seed", range(40))
def test_ids_unique_never_reused_and_consecutive(seed):
    lk = motion.PersonLinker(max_gap=3, max_dist=12, min_joints=3)
    issued, live_last = 0, {}
    for t, recs in enumerate(random_sequence(seed)):
        ids = lk.link(recs)
        assert ids.shape == (len(recs),) and len(set(ids.tolist())) == len(ids)
        new = sorted(i for i in ids if i >= issued)
        assert new == list(range(issued, issued + len(new)))              # new ids consecutive, in person order
        assert [i for i in ids if i >= issued] == new
        for i in ids:
            if i < issued:                                                 # an old id only while its track is live
                assert t - live_last[i] <= 3
            live_last[int(i)] = t
        issued += len(new)


def test_bad_arguments():
    for kw in (dict(max_gap=0, max_dist=1), dict(max_gap=1, max_dist=-1), dict(max_gap=1, max_dist=np.inf),
               dict(max_gap=1, max_dist=1, min_joints=0), dict(max_gap=1, max_dist=1, min_joints=19)):
        with pytest.raises(ValueError):
            motion.PersonLinker(**kw)
    with pytest.raises(ValueError):
        motion.PersonLinker(1, 1).link(np.zeros((2, 60)))


@pytest.fixture(scope="module")
def video(tmp_path_factory):
    import cv2
    path = str(tmp_path_factory.mktemp("vid") / "t.avi")
    w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (160, 120))
    assert w.isOpened()
    rng = np.random.default_rng(0)
    for _ in range(21):
        w.write(cv2.GaussianBlur(rng.integers(0, 256, (120, 160, 3), dtype=np.uint8), (0, 0), 3))
    w.release()
    return path


def decoded(path):
    import cv2
    v = cv2.VideoCapture(path)
    out = []
    while True:
        ok, f = v.read()
        if not ok:
            break
        (x0, y0), (x1, y1) = REC
        out.append(f[y0:y1, x0:x1])
    return out


def test_host_job_writes_tracks_that_reassemble_to_the_records(video, tmp_path):
    import joblib
    logs = []
    out = E.extract_every_person_from_video(video, str(tmp_path / "t.pkl"), REC, fake_body, fake_hand, max_gap=2,
                                            max_dist=60, batch=4, log=logs.append)
    saved = joblib.load(str(tmp_path / "t.pkl"))
    assert set(saved) == {"count", "tracks"} and saved["count"] == 21
    refs = [motion.pose_mats_every_person(f, fake_body, fake_hand) for f in decoded(video)]
    ids = []
    lk = motion.PersonLinker(2, 60)
    for r in refs:
        ids.append(lk.link(r))
    assert len(saved["tracks"]) == 1 + max(int(i.max()) for i in ids if len(i))
    assert any(len(m) > 3 for _, m in saved["tracks"])                      # some persons are followed
    for tid, (first, mat) in enumerate(saved["tracks"]):
        assert mat.dtype == np.float64 and mat.ndim == 3 and mat.shape[1:] == (60, 3)
        frames = [t for t in range(21) if tid in ids[t]]
        assert first == frames[0] and len(mat) == frames[-1] - frames[0] + 1
        for i in range(len(mat)):
            t = first + i
            if tid in ids[t]:
                assert np.array_equal(mat[i], refs[t][list(ids[t]).index(tid)])
            else:
                assert not mat[i].any()                                    # not matched: zero rows
    for name in ("count", "tracks"):
        assert name in out
    assert logs[0] == "t.pkl-0/21" and logs[-1].endswith("t.pkl is saved!")
    two = E.extract_every_person_from_video(video, str(tmp_path / "t2.pkl"), REC, fake_body, fake_hand, max_gap=2,
                                            max_dist=60, batch=4, decode_workers=2, log=lambda s: None)
    assert two["count"] == 21 and len(two["tracks"]) == len(saved["tracks"])
    for (f1, m1), (f2, m2) in zip(saved["tracks"], two["tracks"]):
        assert f1 == f2 and np.array_equal(m1, m2)


def test_host_job_default_gate_and_index_error(video, tmp_path):
    out = E.extract_every_person_from_video(video, str(tmp_path / "d.pkl"), REC, fake_body, fake_hand,
                                            log=lambda s: None)
    lk = motion.PersonLinker(15, 0.1 * (REC[1][1] - REC[0][1]))
    ids = [lk.link(motion.pose_mats_every_person(f, fake_body, fake_hand)) for f in decoded(video)]
    assert len(out["tracks"]) == 1 + max(int(i.max()) for i in ids if len(i))

    def raising(img):
        raise IndexError("index 3 is out of bounds")
    with pytest.raises(IndexError):
        E.extract_every_person_from_video(video, str(tmp_path / "e.pkl"), REC, raising, fake_hand, log=lambda s: None)
    assert not (tmp_path / "e.pkl").exists()
    logs = []
    assert E.extract_every_person_from_video(str(tmp_path / "none.avi"), str(tmp_path / "n.pkl"), REC, fake_body,
                                             fake_hand, log=logs.append) is None
    assert logs and not (tmp_path / "n.pkl").exists()
