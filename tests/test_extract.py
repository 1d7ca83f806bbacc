"""Extraction jobs around the estimators (pytorch_openpose_b200/extract.py; SURVEY.md 8f rows N1/N3/N4): decode ring,
per-frame records, on-disk formats and the resume ledger -- against the reference's own job functions run on the same
synthetic video with the same fake estimators (live, where /root/reference exists) and against themselves."""
import os

import numpy as np
import pytest

from oracle import reference_loader as RL
from pytorch_openpose_b200 import extract as E

live = pytest.mark.skipif(not RL.available(), reason="needs a checkout of the original project (set OPENPOSE_REFERENCE_ROOT)")
REC = [(20, 10), (150, 110)]                      # ROI [(x0, y0), (x1, y1)]


@pytest.fixture(scope="module")
def video(tmp_path_factory):
    import cv2
    path = str(tmp_path_factory.mktemp("vid") / "t.avi")
    w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (160, 120))
    assert w.isOpened()
    rng = np.random.default_rng(0)
    for i in range(21):
        w.write(cv2.GaussianBlur(rng.integers(0, 256, (120, 160, 3), dtype=np.uint8), (0, 0), 3))
    w.release()
    return path


# ---- deterministic fake estimators: results are functions of the pixels they are given ----------------------------
def fake_body(img):
    """Two or three 'persons' whose joints depend on the frame content; some joints missing; one frame with nobody."""
    m = float(img.mean())
    k = int(img[3, 5, 0])
    if k % 7 == 0:
        return np.array([]), -np.ones((0, 20))
    H, W = img.shape[:2]
    n_person = 2 + k % 2
    cand, subset = [], -np.ones((n_person, 20))
    for p in range(n_person):
        for j in range(18):
            if (j + p + k) % 9 == 0:
                continue
            x = (13 * j + 29 * p + k) % (W - 4) + 2
            y = (7 * j + 31 * p + 3 * k) % (H - 4) + 2
            subset[p, j] = len(cand)
            cand.append([float(x), float(y), 0.5 + (m % 1.0) / 4 + j / 100.0, len(cand)])
        subset[p, 18], subset[p, 19] = 10.0 + p, 12
    return np.array(cand), subset


def fake_hand(crop):
    h, w = crop.shape[:2]
    s = int(crop.sum() % 97)
    peaks = np.zeros((21, 3))
    for j in range(21):
        if (j + s) % 5 == 0 or h == 0 or w == 0:
            continue
        peaks[j] = ((3 * j + s) % max(w, 1), (5 * j + s) % max(h, 1), 0.1 + j / 50.0)
    return peaks


class FakePipelinedBody(object):
    """Same results as fake_body through the asynchronous batch interface of `Body`."""
    class _Net(object):
        def session(self):
            return type("S", (), {})()

    def __init__(self):
        self.net = self._Net()

    def submit_batch(self, frames, session, where=0):
        session.out = [fake_body(np.array(f)) for f in frames]

    def collect_batch(self, session):
        return session.out


def test_frame_batches_equal_sequential_decode(video):
    import cv2
    cap = cv2.VideoCapture(video)
    ref = []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        ref.append(f[10:110, 20:150].copy())
    got, firsts = [], []
    for frames, first in E.FrameBatches(video, REC, batch=4, depth=4):
        firsts.append(first)
        got.extend(np.array(frames))                # copy: the ring buffer is reused
    assert E.frame_count(video) == 21 and len(ref) == 21
    assert firsts == [0, 4, 8, 12, 16, 20] and len(got) == 21
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))
    with pytest.raises(FileNotFoundError):
        E.FrameBatches(video + ".missing")
    # several decoders on contiguous segments: same frames, any batch order
    for k in (2, 3, 8):
        seen = {}
        for frames, first in E.FrameBatches(video, REC, batch=4, depth=3, workers=k):
            for f in range(len(frames)):
                seen[first + f] = np.array(frames[f])
        assert sorted(seen) == list(range(21)) and all(np.array_equal(seen[i], ref[i]) for i in range(21))


@pytest.mark.parametrize("mode", ["body", "bodyhand"])
def test_pipelined_extraction_equals_frame_by_frame(video, tmp_path, mode):
    import joblib
    a = E.extract_motion_from_video(video, str(tmp_path / "a.pkl"), REC, fake_body, fake_hand, mode, log=lambda m: None)
    b = E.extract_motion_from_video(video, str(tmp_path / "b.pkl"), REC, FakePipelinedBody(), fake_hand, mode, batch=4,
                                    sessions=3, pinned=False, log=lambda m: None)
    c = E.extract_motion_from_video(video, str(tmp_path / "c.pkl"), REC, FakePipelinedBody(), fake_hand, mode, batch=4,
                                    sessions=2, pinned=False, log=lambda m: None, decode_workers=3)
    assert np.array_equal(a, c)
    assert a.shape == (21, 60 if mode == "bodyhand" else 18, 3) and a.dtype == np.float64
    assert np.array_equal(a, b) and np.array_equal(joblib.load(str(tmp_path / "b.pkl")), a)
    assert (a[:, :18, 2] > 0).any() and (a.reshape(21, -1) == 0).all(1).any()        # people found, and a frame with nobody
    if mode == "bodyhand":
        assert (a[:, 18:, 2] > 0).any()


def test_ledger(tmp_path):
    d = str(tmp_path)
    open(os.path.join(d, "video-001-body.pkl"), "w").close()
    open(os.path.join(d, "notes.txt"), "w").close()
    led = E.ExtractLedger(d)
    assert led.files(init=True) == ["video-001-body.pkl"]
    led.add("video-002-body.pkl")
    assert led.files() == ["video-001-body.pkl\n", "video-002-body.pkl\n"]
    assert led.claimed("video-002-hand.pkl") and not led.claimed("video-003-body.pkl")


@live
def test_ledger_matches_reference(tmp_path):
    rw = RL.load_batch().utilmx.Records_Read_Write()
    d1, d2 = str(tmp_path / "a"), str(tmp_path / "b")
    for d in (d1, d2):
        os.makedirs(d)
        for n in ("video-007-body.pkl", "x.npy", "skip.txt"):
            open(os.path.join(d, n), "w").close()
    led = E.ExtractLedger(d2)
    assert sorted(rw.Get_extract_ed_ing_files(d1, True)) == sorted(led.files(init=True))
    rw.Add_extract_ed_ing_files(d1, "video-008-body.pkl")
    led.add("video-008-body.pkl")
    assert sorted(rw.Get_extract_ed_ing_files(d1)) == sorted(led.files())
    ref_lines = sorted(open(os.path.join(d1, "extract_ed_ing.txt")).read().split())
    assert ref_lines == sorted(open(led.path).read().split())


@live
@pytest.mark.parametrize("mode", ["body", "bodyhand"])
def test_extract_motion_matches_reference_job(video, tmp_path, mode, capsys):
    import joblib
    ME = RL.load_motion_estimation(lambda path: fake_body, lambda path: fake_hand)
    ME.Extract_MotionData_from_Video(video, str(tmp_path / "ref.pkl"), REC, mode)
    ref = joblib.load(str(tmp_path / "ref.pkl"))
    mine = E.extract_motion_from_video(video, str(tmp_path / "mine.pkl"), REC, FakePipelinedBody(), fake_hand, mode,
                                       batch=5, pinned=False)
    assert ref.shape == mine.shape and ref.dtype == mine.dtype and np.array_equal(ref, mine)
    assert np.array_equal(joblib.load(str(tmp_path / "mine.pkl")), ref)


@live
def test_batch_jobs_match_reference_jobs(video, tmp_path):
    import joblib
    import torch
    BME = RL.load_batch_motion_estimation()

    def fake_batch_body(batch):                     # (B,3,h,w) float in [0,1]
        arr = batch.numpy() if hasattr(batch, "numpy") else batch
        return [fake_body(np.round(a.transpose(1, 2, 0) * 255).astype(np.uint8)) for a in arr]

    def fake_batch_hand(batch):
        arr = batch.numpy() if hasattr(batch, "numpy") else batch
        return np.array([fake_hand(np.round(a.transpose(1, 2, 0) * 255).astype(np.uint8)) for a in arr])

    BME.Batch_Body_model = fake_batch_body
    BME.Batch_body_extraction(video, str(tmp_path / "rb.pkl"), 4, REC)
    ref = joblib.load(str(tmp_path / "rb.pkl"))
    mine = E.batch_body_extraction(video, str(tmp_path / "mb.pkl"), 4, REC, fake_batch_body, log=lambda m: None)
    assert ref.shape == (21, 18, 3) and np.array_equal(ref, mine)

    BME.batch_hand_estimation = fake_batch_hand
    BME.Batch_hand_extraction(video, ref, REC, str(tmp_path / "rh.pkl"))
    href = joblib.load(str(tmp_path / "rh.pkl"))
    hmine = E.batch_hand_extraction(video, ref, REC, str(tmp_path / "mh.pkl"), fake_batch_hand, batchsize=32,
                                    log=lambda m: None)
    assert href.shape == (21, 42, 3) and (href[:, :, 2] > 0).any() and np.array_equal(href, hmine)
    # ToTensor equivalence used by both jobs
    from torchvision import transforms
    fr = np.random.default_rng(1).integers(0, 256, (2, 9, 11, 3), dtype=np.uint8)
    assert np.array_equal(E.to_tensor(fr)[1], transforms.ToTensor()(fr[1]).numpy())


@live
def test_combined_dictionary_matches_reference(tmp_path):
    import joblib
    ME = RL.load_motion_estimation(lambda path: fake_body, lambda path: fake_hand)
    d = tmp_path / "data"
    d.mkdir()
    rng = np.random.default_rng(5)
    joblib.dump(rng.random((7, 18, 3)) * 300, str(d / "video-012-body.pkl"))
    joblib.dump(rng.random((5, 60, 3)) * 300, str(d / "video-034-bodyhand.pkl"))
    np.save(str(d / "video-056-body.npy"), rng.random((4, 18, 3)) * 300)
    (d / "readme.txt").write_text("x")
    for mode in ("body", "bodyhand"):
        ME.CombineMotiondata(str(d), str(tmp_path / "ref.pkl"), mode)
        mine = E.combine_motion_data(str(d), str(tmp_path / "mine.pkl"), mode)
        ref = joblib.load(str(tmp_path / "ref.pkl"))
        assert sorted(ref) == sorted(mine) == sorted(joblib.load(str(tmp_path / "mine.pkl")))
        for k in ref:
            assert ref[k][0].dtype == mine[k][0].dtype == np.int16 and ref[k][1].dtype == mine[k][1].dtype == np.float32
            assert np.array_equal(ref[k][0], mine[k][0]) and np.array_equal(ref[k][1], mine[k][1])
    assert len(ref) == 0                           # the reference's bodyhand branch never stores anything


def _job_worker(rank, videofolder, datadir, q):
    import joblib

    def process(videopath, outpath):
        E.batch_body_extraction(videopath, outpath, 4, REC, lambda batch: [
            fake_body(np.round(np.asarray(a).transpose(1, 2, 0) * 255).astype(np.uint8)) for a in batch], log=lambda m: None)

    q.put((rank, E.run_body_job(videofolder, datadir, REC, process, shuffle_seed=rank, log=lambda m: None)))


def test_two_workers_share_a_data_directory(video, tmp_path):
    """One process per GPU, all pointing at the same data directory (srcmx/Batch_motion_Estimation.py:143-163): every
    video is extracted exactly once, the ledger lists each output once, and a later run finds nothing left to do."""
    import multiprocessing as mp
    import shutil
    import joblib
    vids, data = tmp_path / "videos", tmp_path / "data"
    vids.mkdir()
    data.mkdir()
    for k in range(5):
        shutil.copy(video, str(vids / ("%03d-clip.avi" % k)))
    (vids / "notes.txt").write_text("not a video")
    E.ExtractLedger(str(data)).files(init=True)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_job_worker, args=(r, str(vids), str(data), q)) for r in range(2)]
    for p in ps:
        p.start()
    got = dict(q.get(timeout=300) for _ in ps)
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    produced = sorted(got[0] + got[1])
    assert produced == ["video-%03d-body.pkl" % k for k in range(5)]              # disjoint and complete
    ledger = [l.strip() for l in E.ExtractLedger(str(data)).files()]
    assert sorted(ledger) == produced
    ref = E.batch_body_extraction(video, str(tmp_path / "ref.pkl"), 4, REC, lambda batch: [
        fake_body(np.round(np.asarray(a).transpose(1, 2, 0) * 255).astype(np.uint8)) for a in batch], log=lambda m: None)
    for name in produced:
        assert np.array_equal(joblib.load(str(data / name)), ref)
    assert E.run_body_job(str(vids), str(data), REC, lambda a, b: 1 / 0, log=lambda m: None) == []   # nothing left


def test_job_resumes_after_a_worker_died_inside_a_video(tmp_path):
    """A worker that fails after claiming a video must not lock it forever (the reference rebuilds its ledger from the
    files present, srcmx/utilmx.py:190-208, so an unfinished video is redone): the claim goes away with the failure,
    claims left by a dead process are cleared by init=True, and the rerun processes exactly the unfinished videos."""
    import subprocess
    import sys
    vids, data = tmp_path / "videos", tmp_path / "data"
    vids.mkdir()
    data.mkdir()
    for k in range(3):
        (vids / ("%03d-clip.avi" % k)).write_bytes(b"x")
    calls = []

    def process(videopath, outpath):
        calls.append(os.path.basename(videopath))
        if "001" in videopath:
            raise RuntimeError("decoder died")
        with open(outpath, "wb") as f:
            f.write(b"track")

    with pytest.raises(RuntimeError):
        E.run_body_job(str(vids), str(data), REC, process, init=True, log=lambda m: None)
    assert calls == ["000-clip.avi", "001-clip.avi"]
    assert not [f for f in os.listdir(str(data)) if f.endswith(".claim")]          # nothing left locked
    # a worker killed outright (no finally) leaves its claim file: simulate with a claim owned by a dead pid
    dead = subprocess.Popen([sys.executable, "-c", "pass"])
    dead.wait()
    import socket
    (data / ".video-002.claim").write_text("%s %d\n" % (socket.gethostname(), dead.pid))
    # without init the ledger still lists video-001 (appended before processing, like the reference) -> skipped
    calls.clear()
    assert E.run_body_job(str(vids), str(data), REC, process, log=lambda m: None) == []
    # init=True: ledger rebuilt from the files present, stale claims dropped -> 001 fails again, then 002 is done
    calls.clear()
    ok = lambda videopath, outpath: (calls.append(os.path.basename(videopath)), open(outpath, "wb").write(b"track"))
    assert E.run_body_job(str(vids), str(data), REC, ok, init=True, log=lambda m: None) == ["video-001-body.pkl",
                                                                                           "video-002-body.pkl"]
    assert calls == ["001-clip.avi", "002-clip.avi"]
    assert not [f for f in os.listdir(str(data)) if f.endswith(".claim")]
    # a claim held by a LIVE worker on this host survives a rebuild by somebody else
    (vids / "003-clip.avi").write_bytes(b"x")
    live = subprocess.Popen([sys.executable, "-c", "import time; time.sleep(30)"])
    try:
        (data / ".video-003.claim").write_text("%s %d\n" % (socket.gethostname(), live.pid))
        assert E.run_body_job(str(vids), str(data), REC, ok, init=True, log=lambda m: None) == []
    finally:
        live.kill()
        live.wait()
