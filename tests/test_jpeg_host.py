"""The device's JPEG decoder run on the CPU (opb_jpeg_decode_host: the parser, Huffman decoding, ISLOW IDCT, fancy
upsampling and colour conversion the kernels run) equals cv2.imdecode(packet, cv2.IMREAD_COLOR) bit for bit; packets
it does not decode are reported, corrupt ones flagged, malformed headers rejected without a crash."""
import numpy as np
import pytest

from pytorch_openpose_b200 import _lib, jpeg
from tests import jpeg_packets as P


def _ref(pkt, recpoint=None):
    import cv2
    img = cv2.imdecode(pkt, cv2.IMREAD_COLOR)
    assert img is not None
    return img if recpoint is None else img[recpoint[0][1]:recpoint[1][1], recpoint[0][0]:recpoint[1][0]]


@pytest.fixture(scope="module")
def decodable(tmp_path_factory):
    return P.decodable_set(tmp_path_factory.mktemp("jpeg"))


def test_bit_identical_to_imdecode(decodable):
    wrong = []
    for name, pkt in decodable:
        out, status = jpeg.decode_host(pkt)
        if status != 0 or not np.array_equal(out, _ref(pkt)):
            wrong.append(name)
    assert not wrong, "differs from cv2.imdecode: %s" % wrong[:10]
    assert len(decodable) > 200


@pytest.mark.parametrize("quality", [10, 20, 35, 50, 65, 80, 90, 95, 100])
def test_qualities_and_restart_intervals(quality):
    im = P.picture(37, 53, quality)
    for s in P.samplings():
        for rst in (0, 1, 2, 3, 4):
            pkt = P.encode(im, quality, s, rst, rst % 2)
            out, status = jpeg.decode_host(pkt)
            assert status == 0 and np.array_equal(out, _ref(pkt)), (s, rst)


def test_roi_like_frame_batches():
    im = P.picture(61, 90, 3)
    for s in P.samplings():
        pkt = P.encode(im, 70, s)
        for roi in [((0, 0), (90, 61)), ((1, 1), (89, 60)), ((13, 7), (14, 8)), ((80, 50), (200, 300)),
                    ((-10, -5), (-1, -2)), ((0, 0), (1, 61))]:
            out, status = jpeg.decode_host(pkt, roi)
            assert status == 0 and np.array_equal(out, _ref(pkt, roi)), roi


def test_dht_removed_uses_annex_k_tables():
    im = P.picture(40, 56, 5)
    pkt = P.encode(im, 85)
    bare = P.without_dht(pkt)
    assert len(bare) < len(pkt)
    out, status = jpeg.decode_host(bare)
    assert status == 0 and np.array_equal(out, _ref(pkt))


def test_fallback_packets_reported():
    for name, pkt in P.fallback_set():
        out, status = jpeg.decode_host(pkt)
        assert status == jpeg.FALLBACK and out is None, name


def test_exif_orientation_one_is_decoded():
    pkt = P.with_exif_orientation(P.encode(P.picture(20, 30, 1), 80), 1)
    out, status = jpeg.decode_host(pkt)
    assert status == 0 and np.array_equal(out, _ref(pkt))


def test_truncated_packet_flagged():
    pkt = P.encode(P.picture(64, 96, 2), 90)
    scan = [e for m, a, e in P.segments(pkt) if m == 0xDA][0]
    for cut in (scan + 1, (scan + len(pkt)) // 2, len(pkt) - 8):
        out, status = jpeg.decode_host(pkt[:cut])
        assert status == jpeg.CORRUPT, cut


def test_bit_flips_flagged_or_exact():
    """A flipped bit in the entropy data is either found (flagged) or leaves a stream that decodes consistently --
    then libjpeg-turbo decodes it exactly like the device does."""
    import cv2
    pkt = P.encode(P.picture(48, 64, 4), 90)
    scan = [e for m, a, e in P.segments(pkt) if m == 0xDA][0]
    rng = np.random.default_rng(0)
    flagged = 0
    for _ in range(60):
        bad = pkt.copy()
        while True:
            i = int(rng.integers(scan, len(bad) - 2))
            if bad[i] != 0xFF and bad[i - 1] != 0xFF:
                b = bad[i] ^ np.uint8(1 << int(rng.integers(0, 8)))
                if b != 0xFF:
                    bad[i] = b
                    break
        out, status = jpeg.decode_host(bad)
        if status == jpeg.CORRUPT:
            flagged += 1
        else:
            assert status == 0 and np.array_equal(out, cv2.imdecode(bad, cv2.IMREAD_COLOR))
    assert flagged > 0


def _expect_invalid(pkt):
    with pytest.raises(_lib.OpbError) as e:
        jpeg.decode_host(np.frombuffer(bytes(pkt), np.uint8))
    assert e.value.code == _lib.OPB_ERR_INVALID


def test_malformed_headers_invalid():
    pkt = bytes(P.encode(P.picture(16, 16, 0), 80))
    segs = {m: (a, b) for m, a, b in P.segments(np.frombuffer(pkt, np.uint8))}
    _expect_invalid(b"")
    _expect_invalid(b"\x00\x01\x02\x03")
    _expect_invalid(pkt[:2])
    _expect_invalid(pkt[:segs[0xC0][0] + 6])                     # cut inside the frame header
    a, _ = segs[0xDB]
    _expect_invalid(pkt[:a + 4] + bytes([0x07]) + pkt[a + 5:])   # quantisation table slot 7
    a, _ = segs[0xC0]
    _expect_invalid(pkt[:a + 9] + bytes([0]) + pkt[a + 10:])     # zero components
    a, _ = segs[0xC4]
    _expect_invalid(pkt[:a + 5] + bytes([0xFF]) + pkt[a + 6:])   # more codes of length 1 than exist
    _expect_invalid(pkt[:segs[0xC0][0]] + b"\xff\xd9")           # EOI before any frame
    sos, _ = segs[0xDA]
    _expect_invalid(pkt[:segs[0xC0][0]] + pkt[sos:])              # scan without a frame header


def test_capacity():
    pkt = P.encode(P.picture(10, 12, 0), 80)
    h, w, st = _lib.c_int(), _lib.c_int(), _lib.c_int()
    out = np.empty(10, np.uint8)
    rc = _lib.lib().opb_jpeg_decode_host(pkt.ctypes.data, pkt.size, None, out.ctypes.data, out.nbytes,
                                         _lib.ctypes.byref(h), _lib.ctypes.byref(w), _lib.ctypes.byref(st))
    assert rc == _lib.OPB_ERR_CAPACITY and (h.value, w.value) == (10, 12)


def test_device_decode_needs_package_estimators(tmp_path):
    from pytorch_openpose_b200 import extract
    path = str(tmp_path / "c.avi")
    P.write_clip(path, 3, 32, 24, 0)
    with pytest.raises(ValueError):
        extract.batch_body_extraction(path, str(tmp_path / "x.pkl"), 4, None, lambda b: [], log=lambda m: None,
                                      decode="device")
    with pytest.raises(ValueError):
        extract.FrameBatches(path, decode="nvdec")


def test_frame_batches_packets(tmp_path):
    """decode='device' batches carry the clip's raw packets, in order, the last one repeated to pad the last batch."""
    from pytorch_openpose_b200 import extract
    path = str(tmp_path / "c.avi")
    P.write_clip(path, 7, 48, 32, 1)
    pkts = P.clip_packets(path)
    got = []
    for packets, first, n_valid in extract.FrameBatches(path, batch=3, pad_last=True, decode="device"):
        assert len(packets) == 3 and first == len(got)
        got += [packets.packet(i).copy() for i in range(n_valid)]
        assert np.array_equal(packets.packet(2), pkts[min(first + 2, 6)])
    assert len(got) == 7 and all(np.array_equal(a, b) for a, b in zip(got, pkts))
