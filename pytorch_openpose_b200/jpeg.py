"""MJPG frames decoded on the device (csrc/jpeg.cu, opb_jpeg_*).

A decoded frame equals `cv2.imdecode(packet, cv2.IMREAD_COLOR)` bit for bit, ROI-cropped like `extract.FrameBatches`.
Packets the device does not decode (progressive, 4:1:1, EXIF-rotated, ...) and packets whose entropy data turns out
corrupt are decoded with cv2.imdecode and put in their slot, so every frame meets that contract."""
import ctypes
from ctypes import byref, c_int, c_void_p

import numpy as np

from . import _lib

FALLBACK, CORRUPT = _lib.JPEG_FALLBACK, _lib.JPEG_CORRUPT


class Packets(object):
    """A batch of raw JPEG packets: packet i is data[offsets[i]:offsets[i + 1]] (offsets int64, n + 1 entries), to be
    cropped to `recpoint` ((x0, y0), (x1, y1)) or None.  Ordinary host memory: the library parses the packets on the
    host and uploads from its own pinned buffer."""

    def __init__(self, data, offsets, recpoint=None):
        self.data, self.offsets, self.recpoint = data, offsets, recpoint

    @classmethod
    def of(cls, packets, recpoint=None):
        """From a list of byte strings / uint8 arrays (pageable)."""
        arrs = [np.frombuffer(bytes(p), np.uint8) if not isinstance(p, np.ndarray) else p.ravel() for p in packets]
        offsets = np.zeros(len(arrs) + 1, np.int64)
        offsets[1:] = np.cumsum([len(a) for a in arrs])
        data = np.concatenate(arrs) if arrs else np.zeros(0, np.uint8)
        return cls(np.ascontiguousarray(data, np.uint8), offsets, recpoint)

    def __len__(self):
        return len(self.offsets) - 1

    def packet(self, i):
        return self.data[self.offsets[i]:self.offsets[i + 1]]


def _roi(recpoint):
    if recpoint is None:
        return None
    (x0, y0), (x1, y1) = recpoint
    return (c_int * 4)(int(x0), int(y0), int(x1), int(y1))


def _crop(frame, recpoint):
    if recpoint is None:
        return frame
    (x0, y0), (x1, y1) = recpoint
    return frame[y0:y1, x0:x1, :]


def decode_host(packet, recpoint=None):
    """The device's decoder run on the CPU (opb_jpeg_decode_host) -> (frame (h, w, 3) uint8 BGR or None, status);
    status 0, FALLBACK (not decoded: frame None) or CORRUPT (the frame as decoded).  OpbError (OPB_ERR_INVALID) on a
    malformed header."""
    pkt = np.ascontiguousarray(np.frombuffer(bytes(packet), np.uint8) if not isinstance(packet, np.ndarray) else packet,
                               np.uint8).ravel()
    L = _lib.lib()
    roi = _roi(recpoint)
    h, w, st = c_int(), c_int(), c_int()
    _lib.check(L.opb_jpeg_decode_host(pkt.ctypes.data, pkt.size, roi, None, 0, byref(h), byref(w), byref(st)))
    if st.value:
        return None, st.value
    out = np.empty((h.value, w.value, 3), np.uint8)
    _lib.check(L.opb_jpeg_decode_host(pkt.ctypes.data, pkt.size, roi, out.ctypes.data, out.nbytes, byref(h), byref(w),
                                      byref(st)))
    return out, st.value


def host_frame(packet, recpoint, index, shape=None):
    """cv2.imdecode of one packet, ROI-cropped, contiguous; ValueError naming frame `index` if cv2 cannot decode it or
    its size differs from `shape` (h, w) of the batch."""
    import cv2
    img = cv2.imdecode(np.asarray(packet, np.uint8).ravel(), cv2.IMREAD_COLOR)
    if img is None:
        raise ValueError("frame %d: cv2.imdecode cannot decode its JPEG packet" % index)
    img = np.ascontiguousarray(_crop(img, recpoint))
    if shape is not None and img.shape[:2] != tuple(shape):
        raise ValueError("frame %d: decodes to %s, the batch's frames are %s" % (index, img.shape[:2], tuple(shape)))
    return img


class DeviceFrames(object):
    """`packets` decoded on `session`'s stream: `ptr` is the device address of (n, h, w, 3) uint8 BGR frames, valid
    until the session's next decode; `where1` = (ptr, (n, h, w)) is the argument the submits take with where=1.
    Packets the device does not decode are decoded with cv2.imdecode and uploaded before the constructor returns;
    `first` is the index of the batch's first frame (for error messages)."""

    def __init__(self, session, packets, first=0):
        self.session, self.packets, self.first = session, packets, first
        n = len(packets)
        self.flags = np.zeros(n, np.int32)
        ptr, h, w = c_void_p(), c_int(), c_int()
        _lib.check(_lib.lib().opb_jpeg_submit(session.handle, packets.data.ctypes.data, packets.offsets.ctypes.data,
                                              0, n, _roi(packets.recpoint),
                                              self.flags.ctypes.data, byref(ptr), byref(h), byref(w)))
        self.ptr, self.shape = ptr.value, (n, h.value, w.value)
        for i in np.nonzero(self.flags)[0]:
            self._upload(int(i))

    @property
    def where1(self):
        return self.ptr, self.shape

    def _upload(self, i):
        img = host_frame(self.packets.packet(i), self.packets.recpoint, self.first + i, self.shape[1:])
        _lib.check(_lib.lib().opb_jpeg_upload(self.session.handle, i, img.ctypes.data))

    def status(self):
        """Per-frame flags (waits for the decode): FALLBACK / CORRUPT bits."""
        flags = np.zeros(len(self.packets), np.int32)
        _lib.check(_lib.lib().opb_jpeg_status(self.session.handle, flags.ctypes.data))
        return flags

    def repair(self):
        """Waits for the decode; frames the device found corrupt are decoded with cv2.imdecode and uploaded.  True when
        there were any: whatever consumed the frames must run again."""
        bad = np.nonzero((self.status() & CORRUPT) & ~self.flags)[0]
        for i in bad:
            self._upload(int(i))
        return len(bad) > 0

    def fetch(self):
        """The frames on the host (waits for the stream)."""
        out = np.empty(self.shape + (3,), np.uint8)
        _lib.check(_lib.lib().opb_jpeg_fetch(self.session.handle, out.ctypes.data))
        return out


def decode(session, packets, first=0):
    """Frames of `packets` on the device, every one equal to cv2.imdecode's: decode, re-decode corrupt ones on the
    host, (n, h, w, 3) uint8 on the host."""
    d = DeviceFrames(session, packets, first)
    d.repair()
    return d.fetch()
