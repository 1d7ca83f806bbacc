"""`Hand(model_path)(oriImg) -> peaks (21, 3)` -- drop-in for the reference's src/hand.py:16-75 on the GPU."""
import numpy as np

from . import _lib
from .body import _load_checkpoint

DEFAULT_SCALE_SEARCH = (0.5, 1.0, 1.5, 2.0)        # src/hand.py:26


def _is_ragged(crops):
    """A list of crops that do not all share one shape (one that does runs as the equal-size batch it stacks to)."""
    return isinstance(crops, (list, tuple)) and len({np.shape(c) for c in crops}) > 1


def crop_sides(crops):
    """(n,) int32 sides of a list of square (w_i, w_i, 3) crops; raises what Hand()(crop) would raise on an empty crop,
    ValueError on any other shape."""
    sides = np.empty(len(crops), dtype=np.int32)
    for i, c in enumerate(crops):
        shape = np.shape(c)
        if len(shape) != 3 or shape[2] != 3:
            raise ValueError("crop %d: expected an (w, w, 3) uint8 BGR crop, got shape %s" % (i, shape))
        if shape[0] == 0:
            raise ZeroDivisionError("float division by zero")          # src/hand.py:32
        if shape[0] != shape[1]:
            raise ValueError("crop %d is %dx%d: a list of crops of different sizes takes square crops (what "
                             "util.handDetect makes); call Hand()(crop) on a non-square crop" % (i, shape[0], shape[1]))
        sides[i] = shape[0]
    return sides


def pack_crops(crops):
    """List of square (w_i, w_i, 3) uint8 BGR crops -> (packed bytes, offsets (n + 1,) uint64, sides (n,) int32): the
    layout opb_hand_submit_ragged reads, crop i at bytes [offsets[i], offsets[i + 1])."""
    sides = crop_sides(crops)
    offsets = np.zeros(len(crops) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(sides.astype(np.uint64) ** 2 * 3)
    packed = np.concatenate([np.ascontiguousarray(c, dtype=np.uint8).reshape(-1) for c in crops])
    return packed, offsets, sides


class Hand(object):
    def __init__(self, model_path, scale_search=None, device=None):
        weights = model_path if isinstance(model_path, dict) else _load_checkpoint(model_path)
        self.scale_search = list(scale_search) if scale_search is not None else list(DEFAULT_SCALE_SEARCH)
        self.net = _lib.Net(_lib.NET_HAND, weights, device)
        self._session = self.net.session()

    def submit(self, crops, session=None, where=0):
        """crops: (h, w, 3), a batch (n, h, w, 3) of equally sized uint8 BGR crops, or (where 0 only) a list of square
        crops of any sides in pageable host memory (one device pass, row i bit-identical to Hand()(crops[i])).
        where: 0 pageable host array, 1 (device pointer (int), (n, h, w)), 2 pinned host array."""
        s = session or self._session
        sc, ns = _lib.scales_array(self.scale_search)
        if where != 1 and _is_ragged(crops):
            if where != 0:
                raise ValueError("a list of crops of different sides is packed on the host: submit it with where=0")
            packed, offsets, sides = pack_crops(crops)
            s._keepalive = packed
            s._n = len(sides)
            _lib.check(_lib.lib().opb_hand_submit_ragged(s.handle, packed.ctypes.data, offsets.ctypes.data, 0, len(sides),
                                                         sides.ctypes.data, sc, ns))
            return
        if where == 1:
            ptr, (n, h, w) = crops
        else:
            arr = np.ascontiguousarray(crops, dtype=np.uint8)
            if arr.ndim == 3:
                arr = arr[None]
            if arr.shape[1] == 0:
                raise ZeroDivisionError("float division by zero")        # src/hand.py:32
            if arr.ndim != 4 or arr.shape[3] != 3:
                raise ValueError("expected (h, w, 3) or (n, h, w, 3) uint8 BGR crops")
            s._keepalive = arr
            ptr, (n, h, w) = arr.ctypes.data, arr.shape[:3]
        s._n = n
        _lib.check(_lib.lib().opb_hand_submit(s.handle, ptr, where, n, h, w, sc, ns))

    def collect(self, session=None):
        s = session or self._session
        peaks = np.empty((s._n, 21, 3), dtype=np.float64)
        _lib.check(_lib.lib().opb_hand_wait(s.handle, peaks.ctypes.data))
        return peaks

    def last_maps(self, shape, session=None):
        """heatmap_avg (n, h, w, 22) float32 of the last finished batch (src/hand.py:57)."""
        s = session or self._session
        h, w = shape[-3:-1]
        heat = np.empty((s._n, 22, h, w), dtype=np.float32)
        _lib.check(_lib.lib().opb_hand_maps(s.handle, heat.ctypes.data))
        return np.ascontiguousarray(heat.transpose(0, 2, 3, 1))

    MAX_BATCH = 32          # crops per submit: ~0.7 GB of activations per 4-scale crop

    def __call__(self, oriImg):
        """One crop -> (21, 3); a batch (n, h, w, 3) or a list of square crops of any sides -> (n, 21, 3)."""
        ragged = _is_ragged(oriImg)
        if ragged:
            crop_sides(oriImg)              # reject the whole list before any chunk runs
        batched = ragged or np.ndim(oriImg) == 4
        if batched and len(oriImg) > self.MAX_BATCH:
            # large batches (BASELINE config 3: 256 crops) run as chunks, double-buffered over two sessions
            if not hasattr(self, "_session2"):
                self._session2 = self.net.session()
            sessions = (self._session, self._session2)
            out, pending = [], []
            for i, lo in enumerate(range(0, len(oriImg), self.MAX_BATCH)):
                s = sessions[i % 2]
                if len(pending) == 2:
                    out.append(self.collect(pending.pop(0)))
                self.submit(oriImg[lo:lo + self.MAX_BATCH], s)
                pending.append(s)
            for s in pending:
                out.append(self.collect(s))
            return np.concatenate(out, 0)
        self.submit(oriImg)
        peaks = self.collect()
        return peaks if batched else peaks[0]
