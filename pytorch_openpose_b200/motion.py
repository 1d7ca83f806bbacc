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


class PersonLinker(object):
    """Links the persons of consecutive frames into tracks: `link(records)` takes one frame's (P, 60, 3) records (as
    `pose_mats_every_person` returns them) and returns P int track ids.  The rule, exactly (the device tracker,
    `PoseEstimator.tracker`, is held to it bit for bit):

      * Presence: joint j (0-17) of a record is present when its score column is > 0.
      * Track state: each track keeps its id (assigned in creation order from 0, never reused), the 18 body rows of
        the last person it was matched to, and the index of that frame.  A track is live for frame t when
        t - last <= max_gap; a track that is not live at frame t is dropped for good.  Frame indices count every
        linked frame, frames with nobody included.
      * Cost of live track k against person p: J = the joints present in both, ascending.  If |J| < min_joints the
        pair is not eligible.  Otherwise cost = (sum over j in J of sqrt(dx*dx + dy*dy)) / |J| in float64, with
        dx = x_p - x_k, dy = y_p - y_k; every product, sum and the square root rounded separately (no FMA), the sum
        starting at 0.0 and running in joint order.  The pair is eligible when cost <= max_dist.
      * Matching: the eligible pairs sorted by (cost ascending, track id ascending, person index ascending), walked
        greedily; a pair is accepted when neither its track nor its person is taken yet.
      * New tracks: unmatched persons start new tracks, in person-index order.
      * A matched track takes the person's body rows and the frame index.  Hand rows do not enter the cost."""

    def __init__(self, max_gap, max_dist, min_joints=3):
        if int(max_gap) != max_gap or max_gap < 1:
            raise ValueError("max_gap: an int >= 1")
        if not np.isfinite(max_dist) or max_dist < 0:
            raise ValueError("max_dist: a finite number >= 0")
        if int(min_joints) != min_joints or not 1 <= min_joints <= 18:
            raise ValueError("min_joints: an int in 1..18")
        self.max_gap, self.max_dist, self.min_joints = int(max_gap), float(max_dist), int(min_joints)
        self.reset()

    def reset(self):
        """Forget every track: the next frame is frame 0 and the next id is 0."""
        self._ids = np.zeros(0, dtype=np.int64)              # live tracks, ids ascending
        self._rows = np.zeros((0, 18, 3))
        self._last = np.zeros(0, dtype=np.int64)
        self._next = 0
        self._frame = 0

    def link(self, records):
        rec = np.asarray(records, dtype=np.float64)
        if rec.ndim != 3 or rec.shape[1] < 18 or rec.shape[2] != 3:
            raise ValueError("expected (P, 60, 3) records")
        t = self._frame
        live = t - self._last <= self.max_gap
        self._ids, self._rows, self._last = self._ids[live], self._rows[live], self._last[live]
        L, P = len(self._ids), len(rec)
        body = rec[:, :18]
        both = (self._rows[:, None, :, 2] > 0) & (body[None, :, :, 2] > 0)           # (L, P, 18)
        dx = body[None, :, :, 0] - self._rows[:, None, :, 0]
        dy = body[None, :, :, 1] - self._rows[:, None, :, 1]
        dist = np.sqrt(dx * dx + dy * dy)
        total = np.zeros((L, P))
        for j in range(18):                                  # joint order; adding 0.0 for an absent joint is exact
            total = total + np.where(both[:, :, j], dist[:, :, j], 0.0)
        count = both.sum(axis=2)
        ok = count >= self.min_joints
        cost = np.where(ok, total / np.maximum(count, 1), np.inf)
        k, p = np.nonzero(ok & (cost <= self.max_dist))
        c = cost[k, p]
        order = np.lexsort((p, self._ids[k], c))
        ids = np.full(P, -1, dtype=np.int64)
        track_taken = np.zeros(L, dtype=bool)
        for i in order:
            if not track_taken[k[i]] and ids[p[i]] < 0:
                track_taken[k[i]] = True
                ids[p[i]] = self._ids[k[i]]
                self._rows[k[i]] = body[p[i]]
                self._last[k[i]] = t
        new = np.nonzero(ids < 0)[0]
        ids[new] = self._next + np.arange(len(new))
        self._ids = np.concatenate([self._ids, ids[new]])
        self._rows = np.concatenate([self._rows, body[new]])
        self._last = np.concatenate([self._last, np.full(len(new), t, dtype=np.int64)])
        self._next += len(new)
        self._frame = t + 1
        return ids


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

    def collect_every_person(self, pair=None, tracker=None, n_link=None):
        """-> list of n arrays (P_f, 60, 3) float64, equal to `pose_mats_every_person` frame by frame.  Raises IndexError
        like the reference's Body would (src/body.py:173).

        With a `tracker` (`self.tracker(...)`), the first `n_link` frames of the batch (default: all) are linked on the
        device after the hand half, and the result is (records, ids): ids[f] holds the (P_f,) int track ids of frame
        f, -1 for frames past n_link (the padding of a short last batch, which does not advance the tracker).  Batches
        are linked in the order their collects are called; a batch that raises IndexError is not linked."""
        import ctypes
        from . import _lib
        bs, hs = pair or self.sessions(1)[0]
        persons = (ctypes.c_int * bs._batch)()
        status = (ctypes.c_int * bs._batch)()
        if tracker is None:
            _lib.check(_lib.lib().opb_pose_every_wait(bs.handle, persons, status))
        else:
            n_link = bs._batch if n_link is None else int(n_link)
            _lib.check(_lib.lib().opb_pose_every_wait_tracked(bs.handle, tracker.handle, n_link, persons, status))
        counts = list(persons)
        records = np.empty((sum(counts), 60, 3), dtype=np.float64)
        _lib.check(_lib.lib().opb_pose_every_fetch(bs.handle, records.ctypes.data, len(records)))
        split = np.cumsum(counts)[:-1]
        if tracker is None:
            return np.split(records, split)
        ids = np.empty(len(records), dtype=np.int32)
        _lib.check(_lib.lib().opb_pose_every_fetch_ids(bs.handle, ids.ctypes.data, len(ids)))
        return np.split(records, split), np.split(ids.astype(np.int64), split)

    def every_person(self, frames, tracker=None):
        """One frame (H, W, 3) -> (P, 60, 3); a batch (n, H, W, 3) -> list of n such arrays.  With a `tracker`:
        (records, ids) of the same shapes, ids per frame as `collect_every_person` returns them."""
        single = np.ndim(frames) == 3
        self.submit_every_person(np.asarray(frames)[None] if single else frames)
        out = self.collect_every_person(tracker=tracker)
        if tracker is None:
            return out[0] if single else out
        return (out[0][0], out[1][0]) if single else out

    def tracker(self, max_gap, max_dist, min_joints=3):
        """A device tracker for one video (`PersonLinker`'s rule and arguments) on this estimator's GPU, for
        `collect_every_person(..., tracker=)`.  It keeps its tracks until `reset()`."""
        from . import _lib
        return _lib.Tracker(self.body.net.ctx, max_gap, max_dist, min_joints)
