"""JPEG packets the decoder tests share: MJPG clip packets as cv2.VideoWriter writes them, cv2.imencode output over
qualities, sampling factors, restart intervals and optimised tables, grey images, a packet without DHT, and packets
the device must hand to cv2.imdecode (progressive, 4:1:1, 4:4:0, EXIF-rotated)."""
import os
import struct

import numpy as np

ODD_SIZES = [(1, 1), (2, 2), (7, 13), (17, 33), (161, 121), (9, 8), (3, 2)]


def picture(h, w, seed, sigma=6.0):
    """Blurred noise: the detail level of the repository's test clips."""
    import cv2
    a = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    return cv2.GaussianBlur(a, (0, 0), sigma) if min(h, w) > 1 else a


def write_clip(path, n, w, h, seed, sigma=4.0):
    import cv2
    wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (w, h))
    assert wr.isOpened()
    for i in range(n):
        wr.write(picture(h, w, seed + i, sigma))
    wr.release()


def clip_packets(path):
    """The raw JPEG packets of an MJPG clip, in order."""
    import cv2
    cap = cv2.VideoCapture(path)
    cap.set(cv2.CAP_PROP_FORMAT, -1)
    out = []
    while True:
        ok, p = cap.read()
        if not ok:
            break
        out.append(np.array(p, np.uint8).ravel())
    cap.release()
    return out


def encode(img, quality=90, sampling=None, rst=0, optimize=0):
    import cv2
    params = [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_RST_INTERVAL, rst, cv2.IMWRITE_JPEG_OPTIMIZE, optimize]
    if sampling is not None:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sampling]
    ok, pkt = cv2.imencode(".jpg", img, params)
    assert ok
    return pkt.ravel()


def samplings():
    import cv2
    return [cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420]


def segments(pkt):
    """[(marker, start, end)] of the marker segments before the scan (start at the FF byte)."""
    out, i = [], 2
    while i + 4 <= len(pkt) and pkt[i] == 0xFF:
        m = int(pkt[i + 1])
        n = int(pkt[i + 2]) << 8 | int(pkt[i + 3])
        out.append((m, i, i + 2 + n))
        if m == 0xDA:
            break
        i += 2 + n
    return out


def without_dht(pkt):
    """The packet with every DHT segment removed (Motion-JPEG style: the decoder supplies the Annex K tables)."""
    keep = np.ones(len(pkt), bool)
    for m, a, b in segments(pkt):
        if m == 0xC4:
            keep[a:b] = False
    return pkt[keep]


def with_exif_orientation(pkt, orientation):
    """The packet with an APP1 Exif segment (little-endian TIFF, IFD0 holding one Orientation entry) after SOI."""
    tiff = b"II*\x00" + struct.pack("<I", 8) + struct.pack("<H", 1) + struct.pack("<HHIHH", 0x0112, 3, 1, orientation, 0)
    tiff += struct.pack("<I", 0)
    body = b"Exif\x00\x00" + tiff
    app1 = b"\xff\xe1" + struct.pack(">H", len(body) + 2) + body
    return np.frombuffer(bytes(pkt[:2]) + app1 + bytes(pkt[2:]), np.uint8)


def decodable_set(tmpdir, big=True):
    """[(name, packet)] that the device decodes: clips, imencode variants, grey, no DHT."""
    import cv2
    out = []
    clip_sizes = [(1280, 720)] if big else []
    clip_sizes += [(33, 17), (121, 161), (64, 48)]
    for k, (w, h) in enumerate(clip_sizes):
        path = os.path.join(str(tmpdir), "clip%d.avi" % k)
        write_clip(path, 2, w, h, 10 * k)
        out += [("clip %dx%d #%d" % (w, h, i), p) for i, p in enumerate(clip_packets(path))]
    for (h, w) in ODD_SIZES + ([(720, 1280)] if big else []):
        im = picture(h, w, h * 1000 + w)
        for q in (10, 55, 100):
            for s in samplings():
                for rst in (0, 1, 4):
                    out.append(("%dx%d q%d s%x rst%d" % (w, h, q, s, rst), encode(im, q, s, rst)))
        out.append(("%dx%d optimized" % (w, h), encode(im, 75, None, 2, 1)))
        out.append(("%dx%d grey" % (w, h), encode(cv2.cvtColor(im, cv2.COLOR_BGR2GRAY), 80)))
        out.append(("%dx%d grey rst" % (w, h), encode(cv2.cvtColor(im, cv2.COLOR_BGR2GRAY), 30, None, 3)))
        out.append(("%dx%d no DHT" % (w, h), without_dht(encode(im, 85))))
    return out


def fallback_set():
    """[(name, packet)] that the device hands to cv2.imdecode."""
    import cv2
    im = picture(45, 70, 7)
    return [("progressive", np.asarray(cv2.imencode(".jpg", im, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1]).ravel()),
            ("4:1:1", encode(im, 80, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411)),
            ("4:4:0", encode(im, 80, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440)),
            ("exif rotated", with_exif_orientation(encode(im, 80), 6))]
