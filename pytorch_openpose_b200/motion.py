"""Per-frame body + two-hand key-point record (`PoseMat`), the call pattern of the reference's primary caller
(srcmx/MotionEstimation.py:126-216, SURVEY.md 8f row N1) on top of the B200 `Body` / `Hand`.

PoseMat rows: 0-17 body, 18-38 left hand, 39-59 right hand; columns x, y, score; zeros mean "missing"."""
import numpy as np

from . import util


def select_person(candidate, subset):
    """Index of the person with the largest left-shoulder x (srcmx/MotionEstimation.py:144-150); a missing
    shoulder (-1) indexes the LAST candidate, exactly like the reference's candidate[-1]."""
    if len(subset) < 1:
        return None
    xs = np.array([candidate[int(person[5])][0] for person in subset])
    return int(np.argmax(xs))


def pose_mat_every_frame(oriImg, body_estimation, hand_estimation=None, mode="body"):
    """-> (PoseMat (60,3) float64, candidate, subset).  `mode` is 'body' or 'bodyhand'."""
    candidate, subset = body_estimation(oriImg)
    pose = np.zeros((60, 3))
    chosen = select_person(candidate, subset)
    if chosen is not None:
        for k in range(18):
            idx = int(subset[chosen][k])
            if idx != -1:
                pose[k, :] = candidate[idx][:3]
    for i in range(len(subset)):                      # blank the other persons (MotionEstimation.py:160-162)
        if i != chosen:
            subset[i, :] = -1
    if mode == "bodyhand":
        if hand_estimation is None:
            raise ValueError("mode='bodyhand' needs a hand estimator")
        for x, y, w, is_left in util.handDetect(candidate, subset, oriImg):
            crop = oriImg[y:y + w, x:x + w, :]
            if is_left:
                # the hand net detects right hands: mirror, then un-mirror x (MotionEstimation.py:191-194)
                peaks = hand_estimation(np.ascontiguousarray(crop[:, ::-1, :]))
                peaks[:, 0] = np.where(peaks[:, 0] == 0, peaks[:, 0], w - peaks[:, 0] - 1 + x)
                peaks[:, 1] = np.where(peaks[:, 1] == 0, peaks[:, 1], peaks[:, 1] + y)
                pose[18:39, :] = peaks
            else:
                peaks = hand_estimation(crop)
                peaks[:, 0] = np.where(peaks[:, 0] == 0, peaks[:, 0], peaks[:, 0] + x)
                peaks[:, 1] = np.where(peaks[:, 1] == 0, peaks[:, 1], peaks[:, 1] + y)
                pose[39:60, :] = peaks
    return pose, candidate, subset


def pose_mats_every_person(oriImg, body_estimation, hand_estimation):
    """The record of EVERY person `body_estimation` finds: (P, 60, 3) float64, one PoseMat per subset row in subset order.
    Record p is what `pose_mat_every_frame(oriImg, body, hand, 'bodyhand')` returns when its selection picks p: body rows
    from the subset / candidate, `util.handDetect` on that person, `hand_estimation` on each of its boxes (the left crop
    mirrored) and the key points moved into frame coordinates.

    Deviation: a box of width <= 0, on which the reference's Hand raises ZeroDivisionError (src/hand.py:32), gives zero
    hand rows, as on the device (`PoseEstimator.every_person`)."""
    from .extract import _apply_hand
    candidate, subset = body_estimation(oriImg)
    out = np.zeros((len(subset), 60, 3))
    for p in range(len(subset)):
        for k in range(18):
            idx = int(subset[p][k])
            if idx != -1:
                out[p, k, :] = candidate[idx][:3]
        for x, y, w, is_left in util.handDetect(candidate, subset[p:p + 1], oriImg):
            if w <= 0:
                continue
            crop = oriImg[y:y + w, x:x + w, :]
            peaks = hand_estimation(np.ascontiguousarray(crop[:, ::-1, :] if is_left else crop))
            _apply_hand(out[p], peaks, x, y, w, is_left)
    return out


def _frame_batch(bs, frames, where):
    """(pointer, (n, H, W)) of a batch argument: (n, H, W, 3) uint8 host frames (kept alive on the session until the next
    submit) or, for where 1, (device pointer, (n, H, W))."""
    if where == 1:
        return frames
    arr = np.ascontiguousarray(frames, dtype=np.uint8)
    if arr.ndim != 4 or arr.shape[3] != 3:
        raise ValueError("expected an (n, H, W, 3) uint8 BGR array")
    if arr.shape[1] == 0:
        raise ZeroDivisionError("float division by zero")
    bs._keepalive = arr
    return arr.ctypes.data, arr.shape[:3]


class PoseEstimator(object):
    """`MotionData_every_frame(oriImg, mode='bodyhand')` (srcmx/MotionEstimation.py:126-216) for batches of frames with
    everything between the frame upload and PoseMat on the device: body estimation, person selection, `util.handDetect`,
    both hand crops (the left one mirrored) cut out of the frame already in device memory, `Hand` on all crops of the
    batch as ONE ragged launch sequence (every crop keeps its own size), key points moved back to frame coordinates.
    Only PoseMat (n, 60, 3) comes back.  Results equal `pose_mat_every_frame` frame by frame.

    `body` / `hand`: this package's `Body` / `Hand`.  An empty hand box, on which the reference raises
    ZeroDivisionError (src/hand.py:32), gives zero rows instead."""

    def __init__(self, body, hand):
        self.body, self.hand = body, hand
        self._pairs = {}

    def sessions(self, n):
        """n (body session, hand session) pairs kept on the estimators (plans and buffers are expensive to warm up)."""
        have = self.__dict__.setdefault("_session_pairs", [])
        while len(have) < n:
            have.append((self.body.net.session(), self.hand.net.session()))
        return have[:n]

    def submit_batch(self, frames, pair=None, where=0, fixed_boxes=None):
        """frames: (n, H, W, 3) uint8 (where 0 pageable / 2 pinned) or (device pointer, (n, H, W)) (where 1).
        fixed_boxes: optional (n, 2, 3) ints [x, y, w] of the left / right hand box replacing handDetect's."""
        import ctypes
        from . import _lib
        bs, hs = pair or self.sessions(1)[0]
        ptr, (n, H, W) = _frame_batch(bs, frames, where)
        bs._batch = n
        fb = None
        if fixed_boxes is not None:
            fb = np.ascontiguousarray(fixed_boxes, dtype=np.int32).reshape(n, 2, 3)
            bs._keepalive_boxes = fb
        b_arr, nb = _lib.scales_array(self.body.scale_search)
        h_arr, nh = _lib.scales_array(self.hand.scale_search)
        _lib.check(_lib.lib().opb_pose_submit_batch(bs.handle, hs.handle, ptr, where, n, H, W, b_arr, nb, h_arr, nh,
                                                    fb.ctypes.data if fb is not None else None))

    def collect(self, pair=None):
        """-> PoseMat (n, 60, 3) float64.  Raises IndexError like the reference's Body would (src/body.py:173)."""
        import ctypes
        from . import _lib
        bs, hs = pair or self.sessions(1)[0]
        out = np.empty((bs._batch, 60, 3), dtype=np.float64)
        status = (ctypes.c_int * bs._batch)()
        _lib.check(_lib.lib().opb_pose_wait(bs.handle, out.ctypes.data, status))
        return out

    def __call__(self, frames):
        single = np.ndim(frames) == 3
        self.submit_batch(np.asarray(frames)[None] if single else frames)
        out = self.collect()
        return out[0] if single else out

    def submit_every_person(self, frames, pair=None, where=0):
        """Every person of every frame, on the device: frames as for `submit_batch`.  Body, `util.handDetect` on every
        subset row, the hand crops cut from the frames in device memory and run through Hand in fixed chunks of 8."""
        from . import _lib
        bs, hs = pair or self.sessions(1)[0]
        ptr, (n, H, W) = _frame_batch(bs, frames, where)
        bs._batch = n
        b_arr, nb = _lib.scales_array(self.body.scale_search)
        h_arr, nh = _lib.scales_array(self.hand.scale_search)
        _lib.check(_lib.lib().opb_pose_every_submit(bs.handle, hs.handle, ptr, where, n, H, W, b_arr, nb, h_arr, nh))

    def collect_every_person(self, pair=None):
        """-> list of n arrays (P_f, 60, 3) float64, equal to `pose_mats_every_person` frame by frame.  Raises IndexError
        like the reference's Body would (src/body.py:173)."""
        import ctypes
        from . import _lib
        bs, hs = pair or self.sessions(1)[0]
        persons = (ctypes.c_int * bs._batch)()
        status = (ctypes.c_int * bs._batch)()
        _lib.check(_lib.lib().opb_pose_every_wait(bs.handle, persons, status))
        counts = list(persons)
        records = np.empty((sum(counts), 60, 3), dtype=np.float64)
        _lib.check(_lib.lib().opb_pose_every_fetch(bs.handle, records.ctypes.data, len(records)))
        return np.split(records, np.cumsum(counts)[:-1])

    def every_person(self, frames):
        """One frame (H, W, 3) -> (P, 60, 3); a batch (n, H, W, 3) -> list of n such arrays."""
        single = np.ndim(frames) == 3
        self.submit_every_person(np.asarray(frames)[None] if single else frames)
        out = self.collect_every_person()
        return out[0] if single else out
