"""MJPG frames decoded on the device (opb_jpeg_*, jpeg.DeviceFrames) equal cv2.imdecode(packet, cv2.IMREAD_COLOR) bit for
bit, in batches, at ROIs, on two sessions at once, with fallback and corrupt packets; every job with decode="device"
writes the file the same job writes from frames cv2.imdecode decoded from the same packets."""
import joblib
import numpy as np
import pytest

from oracle import openpose_oracle as O
from pytorch_openpose_b200 import extract, jpeg
from tests import jpeg_packets as P

pytestmark = pytest.mark.gpu


def _ref(pkt, roi=None):
    import cv2
    img = cv2.imdecode(np.asarray(pkt), cv2.IMREAD_COLOR)
    return img if roi is None else img[roi[0][1]:roi[1][1], roi[0][0]:roi[1][0]]


@pytest.fixture(scope="module")
def session():
    from pytorch_openpose_b200 import Body
    body = Body(O.make_weights("body", 0), scale_search=[0.5])
    return body.net.session(), body.net.session()


def _by_size(named):
    groups = {}
    for name, pkt in named:
        groups.setdefault(_ref(pkt).shape, []).append((name, pkt))
    return groups


def test_device_frames_equal_imdecode(session, tmp_path):
    wrong = []
    for shape, items in _by_size(P.decodable_set(tmp_path)).items():
        for lo in range(0, len(items), 16):
            chunk = items[lo:lo + 16]
            d = jpeg.DeviceFrames(session[0], jpeg.Packets.of([p for _, p in chunk]))
            assert not d.repair() and not d.status().any()
            out = d.fetch()
            wrong += [name for (name, pkt), o in zip(chunk, out) if not np.array_equal(o, _ref(pkt))]
    assert not wrong, wrong[:10]


def test_rois_at_the_borders(session):
    im = P.picture(75, 131, 9)
    for s in P.samplings():
        pkts = [P.encode(im, 80, s), P.encode(im, 40, s, 2)]
        for roi in [((0, 0), (131, 75)), ((0, 0), (1, 1)), ((130, 74), (131, 75)), ((1, 0), (130, 75)),
                    ((0, 3), (131, 74)), ((-7, -9), (500, 500))]:
            out = jpeg.DeviceFrames(session[0], jpeg.Packets.of(pkts, roi)).fetch()
            for o, p in zip(out, pkts):
                assert np.array_equal(o, _ref(p, roi)), (s, roi)


@pytest.mark.parametrize("batch", [1, 5, 8])
def test_frame_batches_padded_last_batch(session, tmp_path, batch):
    path = str(tmp_path / "c.avi")
    P.write_clip(path, 13, 96, 64, 3)
    pkts = P.clip_packets(path)
    rec = ((5, 3), (90, 60))
    seen = 0
    for packets, first, n_valid in extract.FrameBatches(path, rec, batch=batch, pad_last=True, decode="device"):
        assert len(packets) == batch
        out = jpeg.decode(session[0], packets, first)
        for f in range(batch):
            assert np.array_equal(out[f], _ref(pkts[min(first + f, len(pkts) - 1)], rec))
        seen += n_valid
    assert seen == len(pkts) == 13


def test_two_sessions_in_flight(session):
    a = [P.encode(P.picture(120, 160, k), 85, P.samplings()[k % 3]) for k in range(6)]
    b = [P.encode(P.picture(120, 160, 50 + k), 60, P.samplings()[(k + 1) % 3], k % 3) for k in range(6)]
    da = jpeg.DeviceFrames(session[0], jpeg.Packets.of(a))
    db = jpeg.DeviceFrames(session[1], jpeg.Packets.of(b))
    fb, fa = db.fetch(), da.fetch()
    assert all(np.array_equal(o, _ref(p)) for o, p in zip(fa, a))
    assert all(np.array_equal(o, _ref(p)) for o, p in zip(fb, b))


def test_mixed_fallback_and_corrupt_redo(session):
    im = P.picture(45, 70, 7)
    good = P.encode(im, 80)
    scan = [e for m, a, e in P.segments(good) if m == 0xDA][0]
    corrupt = good.copy()
    corrupt[scan + 3:scan + 40] = 0x00                       # zeros run out of the Huffman codes' reach
    assert jpeg.decode_host(corrupt)[1] == jpeg.CORRUPT
    named = dict(P.fallback_set())
    fallback = [named["progressive"], named["4:1:1"], named["4:4:0"]]
    pkts = [good] + fallback + [corrupt, good]
    d = jpeg.DeviceFrames(session[0], jpeg.Packets.of(pkts))
    assert list(d.flags) == [0, 1, 1, 1, 0, 0]
    assert d.status()[4] & jpeg.CORRUPT
    assert d.repair()
    out = d.fetch()
    for o, p in zip(out, pkts):
        assert np.array_equal(o, _ref(p))
    # an EXIF-rotated packet comes back from cv2.imdecode turned by 90 degrees: it does not fit the batch
    with pytest.raises(ValueError, match="frame 1"):
        jpeg.DeviceFrames(session[0], jpeg.Packets.of([good, named["exif rotated"]]))


def _corrupted(pkt):
    """The packet with a run of zeros early in its scan: the device flags it, cv2.imdecode still decodes it."""
    bad = np.array(pkt, np.uint8).ravel()
    scan = [e for m, a, e in P.segments(bad) if m == 0xDA][0]
    bad[scan + 3:scan + 40] = 0x00
    return bad


class _Capture(object):
    """cv2.VideoCapture over `real`: raw packet `corrupt_at` (when reading packets) is `_corrupted`; with `imdecode`
    it reads packets and returns cv2.imdecode of each -- the frame source decode='device' must match."""

    def __init__(self, real, path, corrupt_at=None, imdecode=False):
        import cv2
        self.c, self.corrupt_at, self.imdecode, self.raw, self.i = real(path), corrupt_at, imdecode, False, 0
        if imdecode:
            self.set(cv2.CAP_PROP_FORMAT, -1)

    def isOpened(self):
        return self.c.isOpened()

    def get(self, prop):
        return self.c.get(prop)

    def set(self, prop, value):
        import cv2
        if prop == cv2.CAP_PROP_FORMAT and value == -1:
            self.raw = True
        return self.c.set(prop, value)

    def read(self):
        import cv2
        ok, p = self.c.read()
        if ok and self.raw:
            if self.i == self.corrupt_at:
                p = _corrupted(p)
            self.i += 1
            if self.imdecode:
                p = cv2.imdecode(p, cv2.IMREAD_COLOR)
        return ok, p

    def release(self):
        self.c.release()


def _both(monkeypatch, run, tmp_path, corrupt_at=None):
    """run(outdir, decode) under decode='device' and under decode='cv2' with frames from cv2.imdecode of the same
    packets (packet `corrupt_at` corrupted in both).  Returns the results of DeviceFrames.repair in the device run."""
    import cv2
    real = cv2.VideoCapture
    (tmp_path / "d").mkdir()
    (tmp_path / "h").mkdir()
    repairs = []
    repair = jpeg.DeviceFrames.repair

    def spy(self):
        repairs.append(repair(self))
        return repairs[-1]
    with monkeypatch.context() as m:
        m.setattr(jpeg.DeviceFrames, "repair", spy)
        m.setattr(cv2, "VideoCapture", lambda path: _Capture(real, path, corrupt_at))
        run(tmp_path / "d", "device")
    with monkeypatch.context() as m:
        m.setattr(cv2, "VideoCapture", lambda path: _Capture(real, path, corrupt_at, imdecode=True))
        run(tmp_path / "h", "cv2")
    return repairs


def _same_files(a, b):
    """Both directories hold the same non-empty set of files with equal contents; -> count of non-zero values."""
    names = sorted(p.name for p in a.iterdir())
    assert names and names == sorted(p.name for p in b.iterdir())
    nonzero = 0
    for name in names:
        x, y = joblib.load(a / name), joblib.load(b / name)
        if isinstance(x, dict):
            assert x["count"] == y["count"] and len(x["tracks"]) == len(y["tracks"])
            for (f0, m0), (f1, m1) in zip(x["tracks"], y["tracks"]):
                assert f0 == f1 and np.array_equal(m0, m1)
                nonzero += int(np.count_nonzero(m0))
        else:
            assert np.array_equal(x, y), name
            nonzero += int(np.count_nonzero(x))
    return nonzero


@pytest.fixture(scope="module")
def clip(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("clip") / "v.avi")
    P.write_clip(path, 11, 160, 120, 21, sigma=3.0)
    return path


REC = ((4, 2), (150, 118))


@pytest.mark.parametrize("mode", ["body", "bodyhand"])
def test_extract_motion_job(monkeypatch, tmp_path, clip, mode):
    from pytorch_openpose_b200 import Body, Hand
    body = Body(O.make_weights("body", 2, "kaiming"), scale_search=[0.5, 1.0])
    hand = Hand(O.make_weights("hand", 5, "kaiming"), scale_search=[0.5, 1.0])
    _both(monkeypatch, lambda d, dec: extract.extract_motion_from_video(
        clip, str(d / "o.pkl"), REC, body, hand, mode, batch=4, sessions=2, log=lambda m: None, decode=dec), tmp_path)
    _same_files(tmp_path / "d", tmp_path / "h")


def test_every_person_job(monkeypatch, tmp_path, clip):
    from pytorch_openpose_b200 import Body, Hand
    body = Body(O.make_weights("body", 2, "kaiming"), scale_search=[0.5, 1.0])
    hand = Hand(O.make_weights("hand", 5, "kaiming"), scale_search=[0.5, 1.0])
    _both(monkeypatch, lambda d, dec: extract.extract_every_person_from_video(
        clip, str(d / "t.pkl"), REC, body, hand, batch=4, log=lambda m: None, decode=dec), tmp_path)
    _same_files(tmp_path / "d", tmp_path / "h")


@pytest.fixture(scope="module")
def batched():
    from pytorch_openpose_b200.batch_model import Batch_body, Batch_hand
    return Batch_body(O.make_weights("body", 2, "kaiming")), Batch_hand(O.make_weights("hand", 5, "kaiming"))


def test_batch_jobs(monkeypatch, tmp_path, clip, batched):
    body, hand = batched

    def run(d, dec):
        m = extract.batch_body_extraction(clip, str(d / "b.pkl"), 4, REC, body, log=lambda m: None, decode=dec)
        track = m.copy()
        track[:, 2] = [50, 40, 0.9]                              # both arms in view: the hand path crops for real
        track[:, 5] = [110, 40, 0.9]
        track[:, 4] = [60, 70, 0.9]
        track[:, 3] = [50, 60, 0.9]
        track[:, 7] = [100, 70, 0.9]
        track[:, 6] = [110, 60, 0.9]
        extract.batch_hand_extraction(clip, track, REC, str(d / "h.pkl"), hand, batchsize=4, log=lambda m: None,
                                      decode=dec)
        extract.batch_bodyhand_extraction(clip, str(d / "bb.pkl"), str(d / "bh.pkl"), 4, REC, body, hand,
                                          log=lambda m: None, decode=dec)
        extract.batch_every_person_extraction(clip, str(d / "e.pkl"), 4, REC, body, hand, log=lambda m: None,
                                              decode=dec)
    assert not any(_both(monkeypatch, run, tmp_path))
    assert _same_files(tmp_path / "d", tmp_path / "h") > 0


def test_job_reruns_a_batch_with_a_corrupt_packet(monkeypatch, tmp_path, clip, batched):
    """One packet of the clip is corrupt: the device flags it, the job decodes it with cv2.imdecode, runs the batch
    again, and writes the file of the job fed cv2.imdecode frames."""
    import cv2
    body, hand = batched
    pkt = _corrupted(P.clip_packets(clip)[6])
    assert jpeg.decode_host(pkt)[1] == jpeg.CORRUPT and cv2.imdecode(pkt, cv2.IMREAD_COLOR) is not None
    track = np.zeros((11, 18, 3))
    track[:, 2] = [50, 40, 0.9]
    track[:, 5] = [110, 40, 0.9]
    track[:, 4] = [60, 70, 0.9]
    track[:, 3] = [50, 60, 0.9]
    track[:, 7] = [100, 70, 0.9]
    track[:, 6] = [110, 60, 0.9]

    def run(d, dec):
        extract.batch_body_extraction(clip, str(d / "b.pkl"), 4, REC, body, log=lambda m: None, decode=dec)
        extract.batch_hand_extraction(clip, track, REC, str(d / "h.pkl"), hand, batchsize=4, log=lambda m: None,
                                      decode=dec)
    assert sum(_both(monkeypatch, run, tmp_path, corrupt_at=6)) == 2
    assert _same_files(tmp_path / "d", tmp_path / "h") > 0


def test_device_frames_feed_the_networks(session, clip, batched):
    """The where=1 submits read the decoded frames: the network maps equal those of the same frames from the host."""
    from pytorch_openpose_b200 import Body
    body_b, _ = batched
    packets = jpeg.Packets.of(P.clip_packets(clip)[:4], REC)
    host = np.ascontiguousarray(np.stack([_ref(p, REC) for p in P.clip_packets(clip)[:4]]))
    s = body_b.net.session()
    d = jpeg.DeviceFrames(s, packets)
    body_b.submit_frames(d.where1, s, where=1)
    body_b.collect(s)
    dev_maps = body_b.last_maps(s)
    body_b.submit_frames(host, s, where=0)
    body_b.collect(s)
    host_maps = body_b.last_maps(s)
    assert np.abs(host_maps[0]).max() > 0
    assert all(np.array_equal(a, b) for a, b in zip(dev_maps, host_maps))
    body = Body(O.make_weights("body", 2, "kaiming"), scale_search=[0.5])
    s = body.net.session()
    d = jpeg.DeviceFrames(s, packets)
    body.submit_batch(d.where1, s, where=1)
    body.collect_batch(s)
    dev_maps = body.last_maps(host.shape, s)
    body.submit_batch(host, s, where=0)
    body.collect_batch(s)
    host_maps = body.last_maps(host.shape, s)
    assert np.abs(host_maps[0]).max() > 0
    assert all(np.array_equal(a, b) for a, b in zip(dev_maps, host_maps))
