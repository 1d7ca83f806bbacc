"""Every person on the batched estimators, host side: extract.batch_pose_mats_every_person (the contract and oracle of
BatchPoseEstimator.every_person) and the fallback of extract.batch_every_person_extraction with estimators other than
this package's Batch_body / Batch_hand."""
import numpy as np
import pytest

from pytorch_openpose_b200 import extract as E
from pytorch_openpose_b200 import motion
from tests.test_batch_bodyhand_job import fake_batch_body, fake_batch_hand
from tests.test_extract import REC
from tests.test_person_linker import decoded


@pytest.fixture(scope="module")
def video(tmp_path_factory):
    import cv2
    path = str(tmp_path_factory.mktemp("vid") / "t.avi")
    w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (160, 120))
    assert w.isOpened()
    rng = np.random.default_rng(3)
    for _ in range(13):
        w.write(cv2.GaussianBlur(rng.integers(0, 256, (120, 160, 3), dtype=np.uint8), (0, 0), 3))
    w.release()
    return path


def one_person_body(batch):
    """fake_batch_body keeping only the first subset row of every frame"""
    return [(c, s[:1]) for c, s in fake_batch_body(batch)]


def test_records_are_the_bodyhand_rows_of_each_person(video):
    frames = np.stack(decoded(video))
    out = E.batch_pose_mats_every_person(frames, fake_batch_body, fake_batch_hand)
    results = fake_batch_body(E.to_tensor(frames))
    assert len(out) == len(frames) and any(len(r) >= 2 for r in out) and any(len(r) == 0 for r in out)
    for f, ((candidate, subset), recs) in enumerate(zip(results, out)):
        assert recs.shape == (len(subset), 60, 3) and recs.dtype == np.float64
        for p in range(len(subset)):
            body = np.zeros((18, 3))
            for k in range(18):
                if int(subset[p][k]) != -1:
                    body[k] = candidate[int(subset[p][k])][:3]
            assert np.array_equal(recs[p, :18], body), (f, p)
            left, lp, right, rp = E.hand_crops_from_pose(frames[f], body)
            peaks = fake_batch_hand(E.to_tensor(np.stack([left, right])))
            assert np.array_equal(recs[p, 18:39], E._box_to_roi(peaks[0], lp, 368, mirrored=True)), (f, p)
            assert np.array_equal(recs[p, 39:60], E._box_to_roi(peaks[1], rp, 368, mirrored=False)), (f, p)
    assert any((r[:, 18:, :2] != 0).any() for r in out)                      # hands inside boxes


def test_one_person_per_frame_equals_the_bodyhand_fallback(video, tmp_path):
    motion_mat, hand_mat = E.batch_bodyhand_extraction(video, str(tmp_path / "b.pkl"), str(tmp_path / "h.pkl"), 4, REC,
                                                       one_person_body, fake_batch_hand, log=lambda s: None)
    out = E.batch_pose_mats_every_person(np.stack(decoded(video)), one_person_body, fake_batch_hand)
    found = 0
    for f, recs in enumerate(out):
        assert len(recs) <= 1
        if len(recs):
            assert np.array_equal(recs[0], np.concatenate([motion_mat[f], hand_mat[f]])), f
            found += 1
        else:
            assert not motion_mat[f].any()
    assert found >= 8


def test_box_of_width_zero_is_a_missing_hand():
    frame = np.random.default_rng(1).integers(0, 256, (60, 80, 3), dtype=np.uint8)
    candidate = np.array([[10.0 + j, 20.0, 0.5, j] for j in range(18)])
    candidate[5, :2] = candidate[6, :2] = candidate[7, :2] = (30.0, 30.0)     # left arm collapsed: a box of width 0
    subset = np.concatenate([np.arange(18.0), [5.0, 18.0]])[None]

    def body(batch):
        return [(candidate, subset) for _ in batch]
    rec = E.batch_pose_mats_every_person(frame[None], body, fake_batch_hand)[0]
    grey = fake_batch_hand(E.to_tensor(np.full((1, 368, 368, 3), 128, np.uint8)))[0]
    assert rec.shape == (1, 60, 3)
    assert not rec[0, 18:39, :2].any() and np.array_equal(rec[0, 18:39, 2], grey[:, 2])   # grey-crop scores, no coordinates


def test_fallback_job_writes_the_linked_records(video, tmp_path):
    import joblib
    logs = []
    out = E.batch_every_person_extraction(video, str(tmp_path / "t.pkl"), 4, REC, fake_batch_body, fake_batch_hand,
                                          max_gap=2, max_dist=60, log=logs.append)
    saved = joblib.load(str(tmp_path / "t.pkl"))
    assert set(saved) == {"count", "tracks"} and saved["count"] == 13
    refs = E.batch_pose_mats_every_person(np.stack(decoded(video)), fake_batch_body, fake_batch_hand)
    lk = motion.PersonLinker(2, 60)
    ids = [lk.link(r) for r in refs]
    assert len(saved["tracks"]) == 1 + max(int(i.max()) for i in ids if len(i))
    for tid, (first, mat) in enumerate(saved["tracks"]):
        frames = [t for t in range(13) if tid in ids[t]]
        assert first == frames[0] and mat.shape == (frames[-1] - frames[0] + 1, 60, 3) and mat.dtype == np.float64
        for i in range(len(mat)):
            t = first + i
            want = refs[t][list(ids[t]).index(tid)] if tid in ids[t] else np.zeros((60, 3))
            assert np.array_equal(mat[i], want), (tid, t)
    assert out["count"] == 13 and logs == ["t.pkl-0/13", "%s is saved!" % (tmp_path / "t.pkl")]
    two = E.batch_every_person_extraction(video, str(tmp_path / "t2.pkl"), 3, REC, fake_batch_body, fake_batch_hand,
                                          max_gap=2, max_dist=60, decode_workers=2, log=lambda s: None)
    assert len(two["tracks"]) == len(saved["tracks"])
    for (f1, m1), (f2, m2) in zip(saved["tracks"], two["tracks"]):
        assert f1 == f2 and np.array_equal(m1, m2)


def test_fallback_job_default_gate_index_error_and_missing_video(video, tmp_path):
    out = E.batch_every_person_extraction(video, str(tmp_path / "d.pkl"), 4, REC, fake_batch_body, fake_batch_hand,
                                          log=lambda s: None)
    lk = motion.PersonLinker(15, 0.1 * (REC[1][1] - REC[0][1]))
    ids = [lk.link(r) for r in E.batch_pose_mats_every_person(np.stack(decoded(video)), fake_batch_body, fake_batch_hand)]
    assert len(out["tracks"]) == 1 + max(int(i.max()) for i in ids if len(i))

    def raising(batch):
        raise IndexError("list assignment index out of range")
    with pytest.raises(IndexError):
        E.batch_every_person_extraction(video, str(tmp_path / "e.pkl"), 4, REC, raising, fake_batch_hand,
                                        log=lambda s: None)
    assert not (tmp_path / "e.pkl").exists()
    logs = []
    assert E.batch_every_person_extraction(str(tmp_path / "none.avi"), str(tmp_path / "n.pkl"), 4, REC, fake_batch_body,
                                           fake_batch_hand, log=logs.append) is None
    assert logs and not (tmp_path / "n.pkl").exists()
