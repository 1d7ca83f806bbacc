"""extract.batch_bodyhand_extraction with estimators other than this package's Batch_body / Batch_hand: it runs
batch_body_extraction and then batch_hand_extraction on the same ROI, and writes exactly the two files (and log lines)
the two jobs write (srcmx/Batch_motion_Estimation.py:19-112)."""
import numpy as np
import pytest

from pytorch_openpose_b200 import extract as E
from tests.test_extract import REC, fake_body, fake_hand


def fake_batch_body(batch):                         # (B, 3, h, w) float in [0, 1], like the reference's DataLoader yields
    return [fake_body(np.round(np.asarray(a).transpose(1, 2, 0) * 255).astype(np.uint8)) for a in batch]


def fake_batch_hand(batch):
    return np.array([fake_hand(np.round(np.asarray(a).transpose(1, 2, 0) * 255).astype(np.uint8)) for a in batch])


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


def test_fallback_writes_the_files_of_the_two_jobs(video, tmp_path):
    import joblib
    one, two = [], []
    m, h = E.batch_bodyhand_extraction(video, str(tmp_path / "b1.pkl"), str(tmp_path / "h1.pkl"), 4, REC, fake_batch_body,
                                       fake_batch_hand, log=one.append)
    m2 = E.batch_body_extraction(video, str(tmp_path / "b2.pkl"), 4, REC, fake_batch_body, log=two.append)
    h2 = E.batch_hand_extraction(video, joblib.load(str(tmp_path / "b2.pkl")), REC, str(tmp_path / "h2.pkl"),
                                 fake_batch_hand, batchsize=4, log=two.append)
    assert m.shape == (13, 18, 3) and h.shape == (13, 42, 3)
    for a, b in (("b1.pkl", "b2.pkl"), ("h1.pkl", "h2.pkl")):
        fa, fb = joblib.load(str(tmp_path / a)), joblib.load(str(tmp_path / b))
        assert fa.shape == fb.shape and fa.dtype == fb.dtype == np.float64 and np.array_equal(fa, fb), a
    assert np.array_equal(m, m2) and np.array_equal(h, h2)
    assert [l.replace("1.pkl", "2.pkl") for l in one] == two
    assert (m[:, :, 2] > 0).any() and (h[:, :21, :2] != 0).any() and (h[:, 21:, :2] != 0).any()     # people and hands


def test_missing_video(tmp_path):
    logs = []
    assert E.batch_bodyhand_extraction(str(tmp_path / "none.avi"), str(tmp_path / "b.pkl"), str(tmp_path / "h.pkl"), 4,
                                       REC, fake_batch_body, fake_batch_hand, log=logs.append) is None
    assert logs and not (tmp_path / "b.pkl").exists() and not (tmp_path / "h.pkl").exists()
