"""Video -> motion-data files: the extraction jobs around the estimators (SURVEY.md 8f rows N1 / N3 / N4).

Mirrors, with the same outputs and on-disk formats:
  * `Extract_MotionData_from_Video`  srcmx/MotionEstimation.py:25-77   -> joblib pkl, float64 (T, 18 | 60, 3)
  * `Batch_body_extraction`          srcmx/Batch_motion_Estimation.py:66-112   -> joblib pkl, float64 (T, 18, 3)
  * `Batch_hand_extraction`          srcmx/Batch_motion_Estimation.py:19-63    -> joblib pkl, float64 (T, 42, 3)
  * `HandImageDataset.__getitem__`   srcmx/Batch_model.py:68-104       (hand crops rebuilt from a saved pose track)
  * the resume ledger `extract_ed_ing.txt`   srcmx/utilmx.py:190-208

What is different is the plumbing: frames are decoded and ROI-cropped by a background thread into a ring of (pinned)
batch buffers while the GPU works on the previous batches, and batches go through `Body.submit_batch` on several
sessions instead of one synchronous call per frame.  The estimators are passed in, so the glue is testable without
a GPU."""
import os
import queue
import threading

import numpy as np

from . import util
from .motion import select_person


# ---- decode (cv2.VideoCapture, like the reference) ----------------------------------------------------------------
def frame_count(videopath):
    import cv2
    video = cv2.VideoCapture(videopath)
    if not video.isOpened():
        return None
    n = int(video.get(cv2.CAP_PROP_FRAME_COUNT))
    video.release()
    return n


def _alloc(shape, dtype, pinned):
    if pinned:
        import torch
        t = torch.empty(shape, dtype=getattr(torch, np.dtype(dtype).name), pin_memory=True)
        return t.numpy(), t
    return np.empty(shape, dtype=dtype), None


class FrameBatches(object):
    """Iterates over (frames (n, H, W, 3) uint8 BGR view, first_index): ROI-cropped frames of a video in batches,
    decoded ahead of the consumer into reusable buffers (pinned when `pinned`).  A yielded buffer stays valid until
    `hold` further batches have been taken.

    workers=1 reads the file front to back like the reference (`video.read()` until it fails) and yields batches in
    order.  workers=k splits the frame range into k contiguous, batch-aligned segments, one `cv2.VideoCapture` and
    one thread each (seek with CAP_PROP_POS_FRAMES); batches then arrive in whatever order they are decoded -- every
    batch carries its first frame index -- and frames past the container's reported count are not read.

    decode="device": the frames are not decoded here.  One thread reads the raw JPEG packets of an MJPG video
    (CAP_PROP_FORMAT = -1) into a ring of buffers (pageable: the library parses the packets on the host and copies
    what it uploads into its own pinned buffer, so `pinned` does not apply), and every batch is a `jpeg.Packets` (with `recpoint`) for
    `jpeg.DeviceFrames` to decode on the session that consumes it; pad_last repeats the last packet, batches come in
    order, `workers` is ignored.  A video that is not MJPG raises ValueError."""

    def __init__(self, videopath, recpoint=None, batch=8, depth=4, pinned=False, workers=1, pad_last=False, ordered=False,
                 decode="cv2"):
        import cv2
        if decode not in ("cv2", "device"):
            raise ValueError("decode must be 'cv2' or 'device', not %r" % (decode,))
        probe = cv2.VideoCapture(videopath)
        if not probe.isOpened():
            raise FileNotFoundError("the file %s is not exist" % videopath)
        self.count = int(probe.get(cv2.CAP_PROP_FRAME_COUNT))
        self.device = decode == "device"
        if self.device:
            fourcc = int(probe.get(cv2.CAP_PROP_FOURCC)) & 0xFFFFFFFF
            if fourcc.to_bytes(4, "little").upper() != b"MJPG":
                probe.release()
                raise ValueError("%s: decode='device' reads MJPG video, this one is %r"
                                 % (videopath, fourcc.to_bytes(4, "little")))
            workers = 1
        probe.release()
        self.videopath, self.recpoint, self.batch, self.pinned = videopath, recpoint, batch, pinned
        # pad_last: a short final batch is filled up with copies of its last frame and yielded at full size as
        # (frames, first, n_valid), so that the estimator never sees a new batch size (= a new CNN plan) at a video's end
        self.pad_last = pad_last
        self.hold = max(depth - 2, 1)
        self.workers = max(1, int(workers))
        # ordered: batches are yielded in frame order whatever the workers -- the segments one after the other, so a
        # later segment decodes only as far as its ring of buffers reaches ahead
        self.ordered = ordered
        self._q = queue.Queue()
        self._qs = [queue.Queue() for _ in range(self.workers)] if ordered else [self._q] * self.workers
        n_batches = -(-self.count // batch)
        per = -(-n_batches // self.workers) * batch
        self._rings = []
        for w in range(self.workers):
            lo = w * per
            hi = None if self.workers == 1 else min((w + 1) * per, self.count)
            if self.workers > 1 and lo >= self.count:
                self._qs[w].put(None)
                self._rings.append(None)
                continue
            ring = {"bufs": None, "free": queue.Queue(), "depth": self.hold + 2}
            self._rings.append(ring)
            threading.Thread(target=self._run_packets if self.device else self._run, args=(w, ring, lo, hi),
                             daemon=True).start()

    def _crop(self, frame):
        if self.recpoint is None:
            return frame
        (x0, y0), (x1, y1) = self.recpoint
        return frame[y0:y1, x0:x1, :]                 # frame[Recpoint[0][1]:Recpoint[1][1], Recpoint[0][0]:Recpoint[1][0]]

    def _run(self, w, ring, lo, hi):
        import cv2
        video = cv2.VideoCapture(self.videopath)
        try:
            if lo:
                video.set(cv2.CAP_PROP_POS_FRAMES, lo)
            index, cur, fill, first = lo, None, 0, lo
            while hi is None or index < hi:
                ret, frame = video.read()
                if ret is False:
                    break
                img = self._crop(frame)
                if ring["bufs"] is None:
                    ring["bufs"] = [_alloc((self.batch,) + img.shape, np.uint8, self.pinned) for _ in range(ring["depth"])]
                    for i in range(ring["depth"]):
                        ring["free"].put(i)
                if cur is None:
                    cur, fill, first = ring["free"].get(), 0, index
                ring["bufs"][cur][0][fill] = img
                fill += 1
                index += 1
                if fill == self.batch:
                    self._qs[w].put((w, cur, fill, first))
                    cur = None
            if cur is not None and fill:
                if self.pad_last:
                    ring["bufs"][cur][0][fill:] = ring["bufs"][cur][0][fill - 1]
                self._qs[w].put((w, cur, fill, first))
            self._qs[w].put(None)
        except BaseException as e:                     # surface decode errors in the consumer
            self._qs[w].put(e)
        finally:
            video.release()

    def _run_packets(self, w, ring, lo, hi):
        import cv2
        from .jpeg import Packets
        video = cv2.VideoCapture(self.videopath)
        try:
            video.set(cv2.CAP_PROP_FORMAT, -1)         # raw packets, not decoded frames
            ring["bufs"] = [None] * ring["depth"]
            ring["packets"] = [None] * ring["depth"]
            for i in range(ring["depth"]):
                ring["free"].put(i)
            index, parts, first = 0, [], 0

            def put(parts, fill, first):
                cur = ring["free"].get()
                if self.pad_last:
                    parts = parts + [parts[-1]] * (self.batch - fill)
                offsets = np.zeros(len(parts) + 1, np.int64)
                offsets[1:] = np.cumsum([len(p) for p in parts])
                if ring["bufs"][cur] is None or len(ring["bufs"][cur][0]) < offsets[-1]:
                    ring["bufs"][cur] = _alloc((int(offsets[-1]) * 5 // 4 + 4096,), np.uint8, False)
                data = ring["bufs"][cur][0]
                for p, o in zip(parts, offsets):
                    data[o:o + len(p)] = p
                ring["packets"][cur] = Packets(data, offsets, self.recpoint)
                self._qs[w].put((w, cur, fill, first))

            while True:
                ret, pkt = video.read()
                if ret is False:
                    break
                if not parts:
                    first = index
                parts.append(np.asarray(pkt, np.uint8).ravel())
                index += 1
                if len(parts) == self.batch:
                    put(parts, len(parts), first)
                    parts = []
            if parts:
                put(parts, len(parts), first)
            self._qs[w].put(None)
        except BaseException as e:
            self._qs[w].put(e)
        finally:
            video.release()

    def _items(self):
        if self.ordered:                               # each worker's batches arrive in order: take the workers in turn
            for q in self._qs:
                yield from iter(q.get, None)
            return
        finished = 0
        while finished < self.workers:
            item = self._q.get()
            if item is None:
                finished += 1
                continue
            yield item

    def __iter__(self):
        held = []
        for item in self._items():
            if isinstance(item, BaseException):
                raise item
            w, cur, fill, first = item
            held.append((w, cur))
            if len(held) > self.hold:                  # the consumer is done with the oldest buffer
                ow, oc = held.pop(0)
                self._rings[ow]["free"].put(oc)
            if self.device:
                batch = self._rings[w]["packets"][cur]
                yield (batch, first, fill) if self.pad_last else (batch, first)
            elif self.pad_last:
                yield self._rings[w]["bufs"][cur][0], first, fill
            else:
                yield self._rings[w]["bufs"][cur][0][:fill], first


def _check_decode(decode, native):
    if decode not in ("cv2", "device"):
        raise ValueError("decode must be 'cv2' or 'device', not %r" % (decode,))
    if decode == "device" and not native:
        raise ValueError("decode='device' decodes on the sessions of this package's estimators; these are not")


def _decoded(session, frames, first, where):
    """A FrameBatches batch as the submits take it: packets (decode='device') are decoded on `session`, the one that
    consumes them -> ((device pointer, (n, h, w)), 1, jpeg.DeviceFrames); host frames pass through -> (frames, where,
    None)."""
    from .jpeg import DeviceFrames, Packets
    if isinstance(frames, Packets):
        d = DeviceFrames(session, frames, first)
        return d.where1, 1, d
    return frames, where, None


def _rerun_corrupt(dec, resubmit):
    """Before a batch's results are read: frames whose entropy data the device found corrupt are decoded with
    cv2.imdecode, put in place, and the batch runs again."""
    if dec is not None and dec.repair():
        resubmit()


def _job_sessions(estimator, n):
    """Sessions (stream + plans + buffers) are expensive to warm up: keep them on the estimator across videos."""
    have = estimator.__dict__.setdefault("_job_sessions", [])
    while len(have) < n:
        have.append(estimator.net.session())
    return have[:n]


# ---- per-frame records ----------------------------------------------------------------------------------------------
def body_pose(candidate, subset):
    """(18,3) key points of the person with the right-most left shoulder (srcmx/MotionEstimation.py:141-158,
    srcmx/Batch_motion_Estimation.py:86-105); zeros when nobody was found."""
    pose = np.zeros((18, 3))
    chosen = select_person(candidate, subset)
    if chosen is not None:
        for k in range(18):
            idx = int(subset[chosen][k])
            if idx != -1:
                pose[k, :] = candidate[idx][:3]
    return pose, chosen


def _hand_jobs(frame, candidate, subset, chosen):
    """srcmx/MotionEstimation.py:160-190: boxes of the chosen person only -> [(crop, x, y, w, is_left)], left crops
    mirrored (the hand net detects right hands)."""
    for i in range(len(subset)):
        if i != chosen:
            subset[i, :] = -1
    jobs = []
    for x, y, w, is_left in util.handDetect(candidate, subset, frame):
        crop = frame[y:y + w, x:x + w, :]
        jobs.append((np.ascontiguousarray(crop[:, ::-1, :]) if is_left else np.ascontiguousarray(crop), x, y, w, is_left))
    return jobs


def _apply_hand(pose60, peaks, x, y, w, is_left):
    """srcmx/MotionEstimation.py:185-194: crop coordinates -> frame coordinates; exact zeros mean "missing"."""
    if is_left:
        peaks[:, 0] = np.where(peaks[:, 0] == 0, peaks[:, 0], w - peaks[:, 0] - 1 + x)
        peaks[:, 1] = np.where(peaks[:, 1] == 0, peaks[:, 1], peaks[:, 1] + y)
        pose60[18:39, :] = peaks
    else:
        peaks[:, 0] = np.where(peaks[:, 0] == 0, peaks[:, 0], peaks[:, 0] + x)
        peaks[:, 1] = np.where(peaks[:, 1] == 0, peaks[:, 1], peaks[:, 1] + y)
        pose60[39:60, :] = peaks


class _HandPool(object):
    """Hand crops of a whole body batch in flight on several sessions of a `Hand` (every crop has its own size, so
    each is its own submit); results are applied in submission order per session."""

    def __init__(self, hand, n):
        self.hand = hand
        self.sessions = _job_sessions(hand, n)
        self.busy = [None] * n
        self.turn = 0

    def _retire(self, i):
        if self.busy[i] is not None:
            pose60, x, y, w, is_left = self.busy[i]
            _apply_hand(pose60, self.hand.collect(self.sessions[i])[0], x, y, w, is_left)
            self.busy[i] = None

    def submit(self, pose60, crop, x, y, w, is_left):
        i = self.turn
        self.turn = (self.turn + 1) % len(self.sessions)
        self._retire(i)
        if crop.shape[0] == 0 or crop.shape[1] == 0:
            raise ZeroDivisionError("float division by zero")            # src/hand.py:32 on an empty box
        self.hand.submit(crop, self.sessions[i])
        self.busy[i] = (pose60, x, y, w, is_left)

    def drain(self):
        for i in range(len(self.sessions)):
            self._retire(i)


def _hands_into(pose60, frame, candidate, subset, chosen, hand_estimation):
    for crop, x, y, w, is_left in _hand_jobs(frame, candidate, subset, chosen):
        _apply_hand(pose60, hand_estimation(crop), x, y, w, is_left)


def extract_motion_from_video(videopath, outpath, recpoint, body_estimation, hand_estimation=None, mode="body",
                              batch=8, sessions=2, pinned=None, log=print, decode_workers=1, stats=None, decode="cv2"):
    """`Extract_MotionData_from_Video` (srcmx/MotionEstimation.py:25-77): MotionMat (count, 18 | 60, 3) float64, dumped
    with joblib to `outpath`.  `body_estimation` is a `Body`: batches of frames are kept in flight on `sessions` of its
    sessions; any other callable `frame -> (candidate, subset)` is called frame by frame.

    decode="device" (MJPG video, this package's `Body`, and in mode 'bodyhand' its `Hand` on the device path): the
    JPEG packets go up and are decoded on the session that consumes them (`jpeg.DeviceFrames`); the frames equal
    cv2.imdecode's, which differ from cv2.VideoCapture's by a few LSB (DESIGN.md section 2)."""
    import joblib
    if mode == "bodyhand" and hand_estimation is None:
        raise ValueError("mode='bodyhand' needs a hand estimator")
    pipelined = hasattr(body_estimation, "submit_batch")
    if pinned is None:
        pinned = pipelined
    native_hand = mode == "bodyhand" and pipelined and hasattr(hand_estimation, "submit") and hasattr(hand_estimation, "net")
    from .body import Body
    from .hand import Hand
    on_device = (native_hand and type(body_estimation) is Body and type(hand_estimation) is Hand
                 and os.environ.get("OPB_HOST_HANDS") is None)
    _check_decode(decode, on_device or (mode == "body" and type(body_estimation) is Body))
    try:
        src = FrameBatches(videopath, recpoint, batch=batch, depth=sessions + 3, pinned=pinned, workers=decode_workers,
                           pad_last=pipelined, decode=decode)
    except FileNotFoundError as e:
        log(str(e))
        return None
    joints = 60 if mode == "bodyhand" else 18
    mat = np.zeros((src.count, joints, 3))
    outname = os.path.split(outpath)[1]
    done = 0
    hand_pool = None
    if on_device:
        # both estimators are this package's: person selection, hand boxes, crops and the hand network stay on the
        # device, PoseMat is the only thing that comes back (motion.PoseEstimator)
        return _extract_bodyhand_on_device(src, outpath, body_estimation, hand_estimation, sessions, pinned, log, stats)
    if native_hand:
        hand_pool = _HandPool(hand_estimation, 4)

    def finish(frames, first, results):
        nonlocal done
        for f, (candidate, subset) in enumerate(results):
            if first + f >= len(mat):                                  # container reported fewer frames than it holds
                break
            pose, chosen = body_pose(candidate, subset)
            mat[first + f, :18, :] = pose
            if mode == "bodyhand" and chosen is not None:
                if hand_pool is not None:
                    for job in _hand_jobs(frames[f], candidate, subset, chosen):
                        hand_pool.submit(mat[first + f], *job)
                else:
                    _hands_into(mat[first + f], frames[f], candidate, subset, chosen, hand_estimation)
            if (first + f) % 100 == 0:
                log("%s-%d/%d" % (outname, first + f, src.count))
            done += 1

    if pipelined:
        import time
        clock = {"decode_wait": 0.0, "submit": 0.0, "collect_wait": 0.0, "records": 0.0}
        ss = _job_sessions(body_estimation, sessions)
        pending = []                                                   # (session, frames, first)

        def retire():
            s, fr, fi, nv, dec, arg, wh = pending.pop(0)
            t = time.perf_counter()
            _rerun_corrupt(dec, lambda: body_estimation.submit_batch(arg, s, where=wh))
            res = body_estimation.collect_batch(s)
            clock["collect_wait"] += time.perf_counter() - t
            t = time.perf_counter()
            finish(fr, fi, res[:nv])
            clock["records"] += time.perf_counter() - t

        it = iter(src)
        while True:
            t = time.perf_counter()
            item = next(it, None)
            clock["decode_wait"] += time.perf_counter() - t
            if item is None:
                break
            frames, first, n_valid = item
            if len(pending) == sessions:
                retire()
            s = next(c for c in ss if all(c is not p[0] for p in pending))
            t = time.perf_counter()
            arg, wh, dec = _decoded(s, frames, first, 2 if pinned else 0)
            body_estimation.submit_batch(arg, s, where=wh)
            clock["submit"] += time.perf_counter() - t
            pending.append((s, frames, first, n_valid, dec, arg, wh))
        while pending:
            retire()
        if stats is not None:
            stats.update(clock)
    else:
        for frames, first in src:
            finish(frames, first, [body_estimation(frames[f]) for f in range(len(frames))])
    if hand_pool is not None:
        hand_pool.drain()
    joblib.dump(mat, outpath)
    log("%s is saved!" % outpath)
    return mat


def _pose_estimator(body_estimation, hand_estimation):
    """The `PoseEstimator` of a Body / Hand pair, kept on the Body (its sessions are expensive to warm up)."""
    from .motion import PoseEstimator
    est = body_estimation.__dict__.setdefault("_pose_estimator", None)
    if est is None or est.hand is not hand_estimation:
        est = body_estimation.__dict__["_pose_estimator"] = PoseEstimator(body_estimation, hand_estimation)
    return est


def _extract_bodyhand_on_device(src, outpath, body_estimation, hand_estimation, sessions, pinned, log, stats):
    """mode='bodyhand' with the per-frame caller on the device: batches of frames in flight on `sessions` (body, hand)
    session pairs; every collect returns PoseMat rows for its batch."""
    import time
    import joblib
    est = _pose_estimator(body_estimation, hand_estimation)
    pairs = est.sessions(sessions)
    mat = np.zeros((src.count, 60, 3))
    outname = os.path.split(outpath)[1]
    clock = {"decode_wait": 0.0, "submit": 0.0, "collect_wait": 0.0, "records": 0.0}
    pending = []

    def retire():
        pair, first, nv, dec, arg, wh = pending.pop(0)
        t = time.perf_counter()
        _rerun_corrupt(dec, lambda: est.submit_batch(arg, pair, where=wh))
        pose = est.collect(pair)
        clock["collect_wait"] += time.perf_counter() - t
        hi = min(first + nv, len(mat))
        if hi > first:
            mat[first:hi] = pose[:hi - first]
        if first % 100 < len(pose):
            log("%s-%d/%d" % (outname, first, src.count))

    it = iter(src)
    while True:
        t = time.perf_counter()
        item = next(it, None)
        clock["decode_wait"] += time.perf_counter() - t
        if item is None:
            break
        frames, first, n_valid = item
        if len(pending) == len(pairs):
            retire()
        pair = next(c for c in pairs if all(c is not p[0] for p in pending))
        t = time.perf_counter()
        arg, wh, dec = _decoded(pair[0], frames, first, 2 if pinned else 0)
        est.submit_batch(arg, pair, where=wh)
        clock["submit"] += time.perf_counter() - t
        pending.append((pair, first, n_valid, dec, arg, wh))
    while pending:
        retire()
    if stats is not None:
        stats.update(clock)
    joblib.dump(mat, outpath)
    log("%s is saved!" % outpath)
    return mat


# ---- every person, tracked ------------------------------------------------------------------------------------------
def _write_tracks(outpath, count, frames):
    """frames: [(first frame index, [(P_f, 60, 3) records], [(P_f,) ids])] in frame order -> the joblib file
    {"count": count, "tracks": [(first_frame, posemat (L, 60, 3) float64), ...]} indexed by track id."""
    import joblib
    seen = {}
    for first, recs, ids in frames:
        for f, (r, i) in enumerate(zip(recs, ids)):
            for p, tid in enumerate(i):
                seen.setdefault(int(tid), []).append((first + f, r[p]))
    tracks = []
    for tid in range(len(seen)):
        rows = seen[tid]
        mat = np.zeros((rows[-1][0] - rows[0][0] + 1, 60, 3))
        for t, r in rows:
            mat[t - rows[0][0]] = r
        tracks.append((rows[0][0], mat))
    out = {"count": count, "tracks": tracks}
    joblib.dump(out, outpath)
    return out


def extract_every_person_from_video(videopath, outpath, recpoint, body_estimation, hand_estimation, max_gap=15,
                                    max_dist=None, min_joints=3, batch=8, sessions=2, decode_workers=1, log=print,
                                    decode="cv2"):
    """Body and hands of every person of a video, linked into per-person tracks (`motion.PersonLinker`'s rule), dumped
    with joblib to `outpath` as {"count": T, "tracks": [(first_frame, posemat (L, 60, 3) float64), ...]}, indexed by
    track id.  A track's PoseMat runs from its first to its last matched frame; frames in between where it was not
    matched are zero rows (the reference's "missing").  Coordinates are in ROI coordinates, like the other jobs.

    max_dist=None means 0.1 x the ROI height: a choice that lets a person move a tenth of the picture between matched
    frames, not a measured optimum.  max_gap: frames a track may go unmatched and still be picked up again.

    With this package's `Body` and `Hand`, batches run on the device (`PoseEstimator.every_person` on `sessions`
    session pairs in flight) and are linked there, in frame order, by one tracker.  With any other estimators the job
    runs `motion.pose_mats_every_person` frame by frame and links with `PersonLinker`.  Both write the same file.
    Frames are linked in order, so with decode_workers > 1 the later segments decode only a few batches ahead.  An
    IndexError from Body is raised before anything is written.  decode="device" (MJPG video, the device path): the
    JPEG packets are decoded on the consuming session, as in `extract_motion_from_video`."""
    from .body import Body
    from .hand import Hand
    from .motion import PersonLinker, pose_mats_every_person
    device = type(body_estimation) is Body and type(hand_estimation) is Hand
    _check_decode(decode, device)
    try:
        src = FrameBatches(videopath, recpoint, batch=batch, depth=sessions + 3, pinned=device, workers=decode_workers,
                           pad_last=device, ordered=True, decode=decode)
    except FileNotFoundError as e:
        log(str(e))
        return None
    outname = os.path.split(outpath)[1]
    frames = []
    if device:
        est = _pose_estimator(body_estimation, hand_estimation)
        pairs = est.sessions(sessions)
        tracker = None
        pending = []

        def retire():
            pair, first, nv, dec, arg, wh = pending.pop(0)
            n_link = max(0, min(nv, src.count - first))
            _rerun_corrupt(dec, lambda: est.submit_every_person(arg, pair, where=wh))
            recs, ids = est.collect_every_person(pair, tracker=tracker, n_link=n_link)
            frames.append((first, recs[:n_link], ids[:n_link]))
            if first % 100 < len(recs):
                log("%s-%d/%d" % (outname, first, src.count))

        for fr, first, n_valid in src:
            if len(pending) == len(pairs):
                retire()
            pair = next(c for c in pairs if all(c is not p[0] for p in pending))
            arg, wh, dec = _decoded(pair[0], fr, first, 2)
            if tracker is None:
                height = dec.shape[1] if dec is not None else fr.shape[1]
                tracker = est.tracker(max_gap, 0.1 * height if max_dist is None else max_dist, min_joints)
            est.submit_every_person(arg, pair, where=wh)
            pending.append((pair, first, n_valid, dec, arg, wh))
        while pending:
            retire()
    else:
        linker = None
        for fr, first in src:
            if linker is None:
                linker = PersonLinker(max_gap, 0.1 * fr.shape[1] if max_dist is None else max_dist, min_joints)
            recs, ids = [], []
            for f in range(min(len(fr), src.count - first)):
                recs.append(pose_mats_every_person(fr[f], body_estimation, hand_estimation))
                ids.append(linker.link(recs[-1]))
                if (first + f) % 100 == 0:
                    log("%s-%d/%d" % (outname, first + f, src.count))
            frames.append((first, recs, ids))
    out = _write_tracks(outpath, src.count, frames)
    log("%s is saved!" % outpath)
    return out


# ---- the batched jobs (srcmx/Batch_motion_Estimation.py) -----------------------------------------------------------
def to_tensor(frames_u8):
    """torchvision `transforms.ToTensor()` on a batch: (n,H,W,3) uint8 -> (n,3,H,W) float32 = value / 255."""
    return np.ascontiguousarray(frames_u8.transpose(0, 3, 1, 2)).astype(np.float32) / np.float32(255)


def batch_body_extraction(videopath, outpath, batch_size, recpoint, batch_body_model, log=print, decode_workers=1,
                          sessions=2, decode="cv2"):
    """`Batch_body_extraction` (srcmx/Batch_motion_Estimation.py:66-112) -> MotionMat (COUNTS, 18, 3).  A `Batch_body`
    of this package is fed the decoded uint8 frames directly (`submit_frames`: ToTensor's /255 on the device) on
    `sessions` sessions; any other callable gets `ToTensor`-ed float batches like the reference's DataLoader yields.
    decode="device" (MJPG video, this package's `Batch_body`): the JPEG packets are decoded on the consuming session
    (`jpeg.DeviceFrames`); frames equal cv2.imdecode's (DESIGN.md section 2)."""
    import joblib
    from .batch_model import Batch_body
    pipelined = hasattr(batch_body_model, "submit_frames")
    _check_decode(decode, type(batch_body_model) is Batch_body)
    try:
        src = FrameBatches(videopath, recpoint, batch=batch_size, depth=sessions + 3 if pipelined else 4, pinned=pipelined,
                           workers=decode_workers, pad_last=pipelined, decode=decode)
    except FileNotFoundError as e:
        log(str(e))
        return None
    outname = os.path.split(outpath)[1]
    mat = np.zeros((src.count, 18, 3))
    count = 0

    def finish(first, results):
        nonlocal count
        for f, (candidate, subset) in enumerate(results):
            if first + f < len(mat):
                mat[first + f] = body_pose(candidate, subset)[0]
            count += 1
            if count % 1000 == 0:
                log("%s-%d/%d" % (outname, count, src.count))

    if pipelined:
        ss = _job_sessions(batch_body_model, sessions)
        pending = []
        def retire():
            s, fi, nv, dec, arg, wh = pending.pop(0)
            _rerun_corrupt(dec, lambda: batch_body_model.submit_frames(arg, s, where=wh))
            finish(fi, batch_body_model.collect(s)[:nv])

        for frames, first, n_valid in src:
            if len(pending) == sessions:
                retire()
            s = next(c for c in ss if all(c is not p[0] for p in pending))
            arg, wh, dec = _decoded(s, frames, first, 2)
            batch_body_model.submit_frames(arg, s, where=wh)
            pending.append((s, first, n_valid, dec, arg, wh))
        while pending:
            retire()
    else:
        for frames, first in src:
            finish(first, batch_body_model(to_tensor(frames)))
    joblib.dump(mat, outpath)
    log("the %s file is saved" % outpath)
    return mat


def pose_person(pose):
    """The one-person (candidate (20, 4), subset (1, 20)) that HandImageDataset builds from a saved (18, 3) pose for
    util.handDetect (srcmx/Batch_model.py:75-82): joint i is missing when Python's sum(pose[i, :]) is 0."""
    subset = np.zeros((1, 20))
    candidate = np.zeros((20, 4))
    for i in range(18):
        subset[0, i] = -1 if sum(pose[i, :]) == 0 else i
        candidate[i, :2] = pose[i, :2]
    return candidate, subset


def hand_crops_from_pose(image, pose, boxsize=368):
    """`HandImageDataset.__getitem__` (srcmx/Batch_model.py:68-104) for one ROI-cropped frame and its saved (18,3) pose:
    -> (LeftHand, leftparams, RightHand, rightparams); images uint8 (boxsize, boxsize, 3), grey (128) when the hand
    is missing, the left one mirrored; params = [x, y, w]."""
    import cv2
    candidate, subset = pose_person(pose)
    left = np.zeros((boxsize, boxsize, 3), dtype=np.uint8) + 128
    right = np.zeros_like(left) + 128
    leftparams, rightparams = np.zeros((3,)), np.zeros((3,))
    for x, y, w, is_left in util.handDetect(candidate, subset, image):
        if not is_left:
            right = cv2.resize(image[y:y + w, x:x + w, :], (boxsize, boxsize), interpolation=cv2.INTER_CUBIC)
            rightparams = np.array([x, y, w])
        else:
            left = cv2.resize(cv2.flip(image[y:y + w, x:x + w, :], 1), (boxsize, boxsize), interpolation=cv2.INTER_CUBIC)
            leftparams = np.array([x, y, w])
    return left, leftparams, right, rightparams


def _box_to_roi(peaks, box, boxsize, mirrored):
    """Key points of a `boxsize`-square hand image back to ROI coordinates (srcmx/Batch_motion_Estimation.py:41-56):
    scale by w / boxsize, then shift by the box origin (and un-mirror x for left hands); coordinates that are exactly 0
    mark missing key points and stay 0.  `box` = [x, y, w] (all zero when the hand was not found)."""
    bx, by, bw = box
    xy = peaks[:, :2] * bw / boxsize
    px, py = xy[:, 0], xy[:, 1]
    moved_x = (bw - px - 1 + bx) if mirrored else (px + bx)
    peaks[:, 0] = np.where(px == 0, px, moved_x)
    peaks[:, 1] = np.where(py == 0, py, py + by)
    return peaks


def batch_hand_extraction(videopath, motiondata, recpoints, outpath, batch_hand_estimation, boxsize=368, batchsize=32,
                          log=print, decode_workers=1, sessions=2, decode="cv2"):
    """`Batch_hand_extraction` (srcmx/Batch_motion_Estimation.py:19-63) -> HandMat (COUNTS, 42, 3): rows 0-20 left hand,
    21-41 right hand, in ROI coordinates; a coordinate of exactly 0 means "missing" and is not offset.

    With this package's `Batch_hand` the whole per-frame work -- boxes from the saved pose, crops, network, ROI
    coordinates -- runs on the device (`Batch_hand.submit_track`): decoded frames go up as uint8 from a pinned ring,
    batches are in flight on `sessions` sessions and HandMat rows are the only thing that comes back (batches of at
    most 32 frames; `decode_workers` as in `batch_body_extraction`).  One deviation from the host path: a hand box of
    width 0, on which the reference's cv2.resize raises, is treated as a missing hand.  OPB_HOST_HANDS=1, or any other
    estimator, takes the host path: crops cut with cv2 and `batch_hand_estimation` called on ToTensor-ed batches.
    decode="device" (MJPG video, the device path): the JPEG packets are decoded on the consuming session."""
    import joblib
    from .batch_model import Batch_hand
    on_device = type(batch_hand_estimation) is Batch_hand and os.environ.get("OPB_HOST_HANDS") is None
    _check_decode(decode, on_device)
    if on_device:
        return _batch_hand_on_device(videopath, motiondata, recpoints, outpath, batch_hand_estimation, boxsize,
                                     min(batchsize, Batch_hand.TRACK_BATCH), log, decode_workers, sessions, decode)
    src = FrameBatches(videopath, recpoints, batch=batchsize, depth=4, pinned=False)
    assert src.count == len(motiondata)
    mat = np.zeros((len(motiondata), 42, 3))
    count = 0
    for frames, first in src:
        items = [hand_crops_from_pose(frames[f], motiondata[first + f], boxsize) for f in range(len(frames))]
        lefts = batch_hand_estimation(to_tensor(np.stack([it[0] for it in items])))
        rights = batch_hand_estimation(to_tensor(np.stack([it[2] for it in items])))
        for i, (_, left_box, _, right_box) in enumerate(items):
            mat[count, 21:, :] = _box_to_roi(rights[i], right_box, boxsize, mirrored=False)
            mat[count, :21, :] = _box_to_roi(lefts[i], left_box, boxsize, mirrored=True)
            count += 1
            if count % 1000 == 0:
                log("%s-%d/%d" % (outpath, count, len(motiondata)))
    joblib.dump(mat, outpath)
    log("the %s file is saved" % outpath)
    return mat


def _batch_hand_on_device(videopath, motiondata, recpoints, outpath, est, boxsize, batchsize, log, decode_workers,
                          sessions, decode="cv2"):
    import joblib
    src = FrameBatches(videopath, recpoints, batch=batchsize, depth=sessions + 3, pinned=True, workers=decode_workers,
                       pad_last=True, decode=decode)
    assert src.count == len(motiondata)
    motiondata = np.asarray(motiondata, dtype=np.float64)
    mat = np.zeros((len(motiondata), 42, 3))
    ss = _job_sessions(est, sessions)
    pending = []                                                   # (session, first, n_valid)
    count = 0

    def retire():
        nonlocal count
        s, first, nv, dec, arg, wh, poses = pending.pop(0)
        _rerun_corrupt(dec, lambda: est.submit_track(arg, poses, s, where=wh, boxsize=boxsize))
        hi = min(first + nv, len(mat))
        mat[first:hi] = est.collect_track(s)[:hi - first]
        for _ in range(hi - first):
            count += 1
            if count % 1000 == 0:
                log("%s-%d/%d" % (outpath, count, len(motiondata)))

    for frames, first, n_valid in src:
        nv = max(0, min(n_valid, len(motiondata) - first))
        poses = np.empty((len(frames), 18, 3))
        poses[:nv] = motiondata[first:first + nv]
        poses[nv:] = motiondata[first + nv - 1] if nv else 0         # padded frames: a copy of the last valid pose
        if len(pending) == sessions:
            retire()
        s = next(c for c in ss if all(c is not p[0] for p in pending))
        arg, wh, dec = _decoded(s, frames, first, 2)
        est.submit_track(arg, poses, s, where=wh, boxsize=boxsize)
        pending.append((s, first, nv, dec, arg, wh, poses))
    while pending:
        retire()
    joblib.dump(mat, outpath)
    log("the %s file is saved" % outpath)
    return mat


def batch_bodyhand_extraction(videopath, body_outpath, hand_outpath, batch_size, recpoint, batch_body_model,
                              batch_hand_estimation, boxsize=368, log=print, decode_workers=1, sessions=2, decode="cv2"):
    """`Batch_body_extraction` and then `Batch_hand_extraction` on its track (srcmx/Batch_motion_Estimation.py:19-112)
    -> (MotionMat (COUNTS, 18, 3), HandMat (COUNTS, 42, 3)), written to `body_outpath` / `hand_outpath` with the same
    shapes, dtypes and log lines as `batch_body_extraction` and `batch_hand_extraction`.

    With this package's `Batch_body` and `Batch_hand` the video is decoded once: every batch of frames goes up once from
    a pinned ring and `BatchPoseEstimator` runs body, person selection, hand boxes, crops and the hand network on it in
    one launch sequence, with batches in flight on `sessions` (body, hand) session pairs (at most 32 frames per batch;
    `decode_workers` as in `batch_body_extraction`).  Both tracks equal the two-pass job's bit for bit; a frame on which
    Batch_body raises IndexError makes the job raise it before any file is written.  With any other estimators the two
    jobs run one after the other on the same ROI.

    From `run_body_job`, one video per call, writing the `-hand` track next to the body track:

        def process_video(videopath, outpath):
            batch_bodyhand_extraction(videopath, outpath, outpath.replace("-body.pkl", "-hand.pkl"), 32, recpoint,
                                      Batch_body(body_model_path), Batch_hand(hand_model_path))
        run_body_job(videofolder, datadir, recpoint, process_video)

    (create the two estimators once, outside the closure: their sessions are kept across videos).  decode="device"
    (MJPG video, this package's estimators): the JPEG packets are decoded on the consuming session."""
    from .batch_model import Batch_body, Batch_hand, BatchPoseEstimator
    native = type(batch_body_model) is Batch_body and type(batch_hand_estimation) is Batch_hand
    _check_decode(decode, native)
    if not native:
        motion = batch_body_extraction(videopath, body_outpath, batch_size, recpoint, batch_body_model, log=log,
                                       decode_workers=decode_workers, sessions=sessions)
        if motion is None:
            return None
        hand = batch_hand_extraction(videopath, motion, recpoint, hand_outpath, batch_hand_estimation, boxsize=boxsize,
                                     batchsize=batch_size, log=log, decode_workers=decode_workers, sessions=sessions)
        return motion, hand
    import joblib
    batch = min(batch_size, BatchPoseEstimator.MAX_BATCH)
    try:
        src = FrameBatches(videopath, recpoint, batch=batch, depth=sessions + 3, pinned=True, workers=decode_workers,
                           pad_last=True, decode=decode)
    except FileNotFoundError as e:
        log(str(e))
        return None
    est = _batch_pose_estimator(batch_body_model, batch_hand_estimation)
    pairs = est.sessions(sessions)
    outname = os.path.split(body_outpath)[1]
    motion = np.zeros((src.count, 18, 3))
    hand = np.zeros((src.count, 42, 3))
    pending = []                                                   # (pair, first, n_valid)
    counts = [0, 0]                                                # frames retired: body job, hand job

    def retire():
        pair, first, nv, dec, arg, wh = pending.pop(0)
        _rerun_corrupt(dec, lambda: est.submit(arg, pair, where=wh, boxsize=boxsize))
        m, h = est.collect(pair)
        hi = min(first + nv, len(motion))
        motion[first:hi] = m[:hi - first]
        hand[first:hi] = h[:hi - first]
        for f in range(nv):                                        # the progress lines of the two jobs
            counts[0] += 1
            if counts[0] % 1000 == 0:
                log("%s-%d/%d" % (outname, counts[0], src.count))
            if first + f < hi:
                counts[1] += 1
                if counts[1] % 1000 == 0:
                    log("%s-%d/%d" % (hand_outpath, counts[1], src.count))

    for frames, first, n_valid in src:
        if len(pending) == len(pairs):
            retire()
        pair = next(c for c in pairs if all(c is not p[0] for p in pending))
        arg, wh, dec = _decoded(pair[0], frames, first, 2)
        est.submit(arg, pair, where=wh, boxsize=boxsize)
        pending.append((pair, first, n_valid, dec, arg, wh))
    while pending:
        retire()
    joblib.dump(motion, body_outpath)
    log("the %s file is saved" % body_outpath)
    joblib.dump(hand, hand_outpath)
    log("the %s file is saved" % hand_outpath)
    return motion, hand


def _batch_pose_estimator(batch_body_model, batch_hand_estimation):
    """The `BatchPoseEstimator` of a Batch_body / Batch_hand pair, kept on the Batch_body (its sessions are expensive to
    warm up)."""
    from .batch_model import BatchPoseEstimator
    est = batch_body_model.__dict__.setdefault("_batch_pose_estimator", None)
    if est is None or est.hand is not batch_hand_estimation:
        est = batch_body_model.__dict__["_batch_pose_estimator"] = BatchPoseEstimator(batch_body_model,
                                                                                      batch_hand_estimation)
    return est


# ---- every person on the batched estimators, tracked ----------------------------------------------------------------
def _batch_hand_crops(frame, body, boxsize):
    """`hand_crops_from_pose` on a record's body rows, except that a box of width 0 -- on which cv2.resize raises --
    is a missing hand (grey crop, params 0), as in `Batch_hand.track`."""
    pose = np.array(body, dtype=np.float64)
    candidate, subset = pose_person(pose)
    for x, y, w, is_left in util.handDetect(candidate, subset, frame):
        if w <= 0:
            pose[7 if is_left else 4] = 0                          # drop the wrist: that hand has no box
    return hand_crops_from_pose(frame, pose, boxsize)


def batch_pose_mats_every_person(frames_u8, batch_body_model, batch_hand_estimation, boxsize=368):
    """Every person of every frame on the batched estimators: (n, h, w, 3) uint8 ROI-cropped frames -> list of n arrays
    (P_f, 60, 3) float64, one record per subset row of `batch_body_model`'s result, in subset order.

    Record p of frame f is the row of [MotionMat | HandMat] that `batch_bodyhand_extraction` would write for frame f had
    its person selection picked subset row p:
      * rows 0-17: candidate[subset[p][k]][:3], zero where the index is -1 (as `body_pose`);
      * rows 18-38 (left hand) and 39-59 (right hand): `hand_crops_from_pose(frame, rows 0-17, boxsize)`,
        `batch_hand_estimation` on the ToTensor-ed crops, `_box_to_roi` back to ROI coordinates.
    Every person always gets both crops: a missing hand gets the grey crop and keeps the scores Batch_hand finds on it
    (coordinates 0), as HandImageDataset does.  The records have PoseMat's layout, so `motion.PersonLinker` and the
    tracks file of `extract_every_person_from_video` apply unchanged.

    Deviation (as `Batch_hand.track`): a box of width 0, on which cv2.resize raises, is a missing hand.  A frame on which
    Batch_body raises IndexError raises for the batch.  Works with any estimators: it is the host fallback of
    `batch_every_person_extraction` and the oracle of `BatchPoseEstimator.every_person`."""
    frames_u8 = np.asarray(frames_u8)
    results = batch_body_model(to_tensor(frames_u8)) if len(frames_u8) else []
    out, crops, slots = [], [], []                                 # slots: (frame, person, params, left)
    for f, (candidate, subset) in enumerate(results):
        recs = np.zeros((len(subset), 60, 3))
        for p in range(len(subset)):
            for k in range(18):
                idx = int(subset[p][k])
                if idx != -1:
                    recs[p, k, :] = candidate[idx][:3]
            left, leftparams, right, rightparams = _batch_hand_crops(frames_u8[f], recs[p, :18], boxsize)
            crops += [left, right]
            slots += [(f, p, leftparams, True), (f, p, rightparams, False)]
        out.append(recs)
    for lo in range(0, len(crops), 64):
        peaks = batch_hand_estimation(to_tensor(np.stack(crops[lo:lo + 64])))
        for (f, p, params, left), pk in zip(slots[lo:lo + 64], peaks):
            row = 18 if left else 39
            out[f][p, row:row + 21, :] = _box_to_roi(np.array(pk, dtype=np.float64), params, boxsize, mirrored=left)
    return out


def batch_every_person_extraction(videopath, outpath, batch_size, recpoint, batch_body_model, batch_hand_estimation,
                                  max_gap=15, max_dist=None, min_joints=3, boxsize=368, log=print, decode_workers=1,
                                  sessions=2, decode="cv2"):
    """Body and hands of every person of a video on the batched estimators, linked into per-person tracks
    (`motion.PersonLinker`'s rule), dumped with joblib to `outpath` in the format of `extract_every_person_from_video`:
    {"count": frames, "tracks": [(first_frame, posemat (L, 60, 3) float64), ...]}, indexed by track id, with zero rows
    where a track was not matched.  The records are those of `batch_pose_mats_every_person`, in ROI coordinates.
    max_dist=None means 0.1 x the ROI height; max_gap as in `extract_every_person_from_video`.

    With this package's `Batch_body` and `Batch_hand`, batches of at most `BatchPoseEstimator.MAX_BATCH` frames run on the
    device (`BatchPoseEstimator.every_person`, `sessions` session pairs in flight, frames from a pinned ring) and are
    linked there, in frame order, by one tracker.  With any other estimators the job runs `batch_pose_mats_every_person`
    on batches of `batch_size` frames and links with `PersonLinker`.  Both write the same file and log lines.  Frames are
    linked in order, so with decode_workers > 1 the later segments decode only a few batches ahead.  An IndexError from
    Batch_body is raised before anything is written.

    From `run_body_job`, one video per call:

        body, hand = Batch_body(body_model_path), Batch_hand(hand_model_path)

        def process_video(videopath, outpath):
            batch_every_person_extraction(videopath, outpath, 32, recpoint, body, hand)
        run_body_job(videofolder, datadir, recpoint, process_video, mode="tracks")

    (create the two estimators once, outside the closure: their sessions are kept across videos).  decode="device"
    (MJPG video, this package's estimators): the JPEG packets are decoded on the consuming session."""
    from .batch_model import Batch_body, Batch_hand, BatchPoseEstimator
    from .motion import PersonLinker
    device = type(batch_body_model) is Batch_body and type(batch_hand_estimation) is Batch_hand
    _check_decode(decode, device)
    batch = min(batch_size, BatchPoseEstimator.MAX_BATCH) if device else batch_size
    try:
        src = FrameBatches(videopath, recpoint, batch=batch, depth=sessions + 3 if device else 4, pinned=device,
                           workers=decode_workers, pad_last=device, ordered=True, decode=decode)
    except FileNotFoundError as e:
        log(str(e))
        return None
    outname = os.path.split(outpath)[1]
    frames = []

    def progress(first, n):
        for t in range(first, first + n):
            if t % 100 == 0:
                log("%s-%d/%d" % (outname, t, src.count))

    if device:
        est = _batch_pose_estimator(batch_body_model, batch_hand_estimation)
        pairs = est.sessions(sessions)
        tracker = None
        pending = []                                               # (pair, first, n_valid)

        def retire():
            pair, first, nv, dec, arg, wh = pending.pop(0)
            n_link = max(0, min(nv, src.count - first))
            _rerun_corrupt(dec, lambda: est.submit_every_person(arg, pair, where=wh, boxsize=boxsize))
            recs, ids = est.collect_every_person(pair, tracker=tracker, n_link=n_link)
            frames.append((first, recs[:n_link], ids[:n_link]))
            progress(first, n_link)

        for fr, first, n_valid in src:
            if len(pending) == len(pairs):
                retire()
            pair = next(c for c in pairs if all(c is not p[0] for p in pending))
            arg, wh, dec = _decoded(pair[0], fr, first, 2)
            if tracker is None:
                height = dec.shape[1] if dec is not None else fr.shape[1]
                tracker = est.tracker(max_gap, 0.1 * height if max_dist is None else max_dist, min_joints)
            est.submit_every_person(arg, pair, where=wh, boxsize=boxsize)
            pending.append((pair, first, n_valid, dec, arg, wh))
        while pending:
            retire()
    else:
        linker = None
        for fr, first in src:
            if linker is None:
                linker = PersonLinker(max_gap, 0.1 * fr.shape[1] if max_dist is None else max_dist, min_joints)
            n = max(0, min(len(fr), src.count - first))
            recs = batch_pose_mats_every_person(fr[:n], batch_body_model, batch_hand_estimation, boxsize)
            frames.append((first, recs, [linker.link(r) for r in recs]))
            progress(first, n)
    out = _write_tracks(outpath, src.count, frames)
    log("%s is saved!" % outpath)
    return out


# ---- resume ledger (srcmx/utilmx.py:190-208) ----------------------------------------------------------------------
class ExtractLedger(object):
    """`extract_ed_ing.txt` in the data directory: one output file name per line, appended BEFORE a video is processed
    so that several workers (one per GPU) sharing the directory skip each other's videos."""
    NAME = "extract_ed_ing.txt"

    def __init__(self, datadir):
        self.path = os.path.join(datadir, self.NAME)
        self.datadir = datadir

    def files(self, init=False):
        """init=True rebuilds the ledger from the .npy / .pkl files present; entries keep their trailing newline when
        read back, exactly like the reference's readlines()."""
        if init:
            names = [f for f in os.listdir(self.datadir) if os.path.splitext(f)[1] in (".npy", ".pkl")]
            self._drop_stale_claims(names)
            with open(self.path, "w") as f:
                for name in names:
                    f.write("%s\n" % name)
            return names
        with open(self.path, "r") as f:
            return f.readlines()

    def add(self, name):
        with open(self.path, "a") as f:
            f.write("%s\n" % name)

    # ---- claim files: `.video-XXX.claim` holding "host pid" of the worker that took the video ----
    def claim_path(self, outname):
        return os.path.join(self.datadir, "." + outname[:9] + ".claim")

    def try_claim(self, outname):
        """Atomically take a video: only one worker creates the claim file."""
        import socket
        try:
            fd = os.open(self.claim_path(outname), os.O_CREAT | os.O_EXCL | os.O_WRONLY)
        except FileExistsError:
            return False
        with os.fdopen(fd, "w") as f:
            f.write("%s %d\n" % (socket.gethostname(), os.getpid()))
        return True

    def release(self, outname):
        try:
            os.remove(self.claim_path(outname))
        except FileNotFoundError:
            pass

    def _drop_stale_claims(self, present):
        """A rebuild of the ledger (init=True) re-opens every video without an output file, like the reference's
        (srcmx/utilmx.py:190-208): claims left behind by a worker that died are removed.  A claim whose owner is a live
        process on this host is kept (that worker is still busy with the video)."""
        import socket
        have = set(n[:9] for n in present)
        for f in os.listdir(self.datadir):
            if not (f.startswith(".") and f.endswith(".claim")):
                continue
            if f[1:10] in have:
                continue
            path = os.path.join(self.datadir, f)
            try:
                with open(path) as fh:
                    host, pid = fh.read().split()
                if host == socket.gethostname() and int(pid) != os.getpid():
                    os.kill(int(pid), 0)                 # raises if the owner is gone
                    continue
            except (OSError, ValueError):
                pass
            try:
                os.remove(path)
            except FileNotFoundError:
                pass

    def claimed(self, outname):
        """The reference's test: the first 9 characters ('video-XXX') of any ledger line (Batch_motion_Estimation.py:156)."""
        return outname[:9] in [x[:9] for x in self.files()]


# ---- combined dictionary (srcmx/MotionEstimation.py:307-341) ---------------------------------------------------------
def combine_motion_data(datafolder, outpath, mode, pattern=r"\d+"):
    """`CombineMotiondata`: every .npy / .pkl track in `datafolder` under the first number in its file name ->
    {key: (positions int16 (T,18,2), scores float32 (T,18))}, dumped with joblib.  Like the reference, mode
    'bodyhand' converts the tracks but stores nothing (the assignment is missing at MotionEstimation.py:336-340), so
    its dictionary is empty; files whose key was already taken are skipped in os.listdir order."""
    import re
    import joblib
    out = {}
    for filename in os.listdir(datafolder):
        ext = os.path.splitext(filename)[1]
        key = re.findall(pattern, filename)
        if len(key) == 0 or key[0] in out:
            continue
        if ext not in (".npy", ".pkl"):
            continue
        path = os.path.join(datafolder, filename)
        data = np.load(path) if ext == ".npy" else joblib.load(path)
        if mode == "body":
            out[key[0]] = (data[:, :18, :2].astype(np.int16), data[:, :18, -1].astype(np.float32))
    joblib.dump(out, outpath)
    return out


# ---- the per-directory job loop (srcmx/Batch_motion_Estimation.py:143-163), one worker per GPU ----------------------
VIDEO_EXTENSIONS = (".mp4", ".mkv", ".rmvb", ".avi")


def run_body_job(videofolder, datadir, recpoint, process_video, mode="body", init=False, shuffle_seed=None, log=print):
    """Every video of `videofolder` that nobody has claimed yet -> `datadir/video-XXX-<mode>.pkl` (XXX = first three
    characters of the file name), exactly the loop of `Test(code=0)`: the output name is appended to the ledger BEFORE
    the video is processed, and a name whose first nine characters are already in the ledger is skipped.  Several
    workers (one process per GPU) may share `datadir`; the reference relies on shuffling to keep them apart, here a
    claim is additionally made atomic with an exclusive claim file next to the ledger (removed when the video is done
    or has failed; stale ones are cleared by init=True), so two workers never take the same video.  `process_video(videopath, outpath)` does the work (e.g. a lambda around `batch_body_extraction`).
    Returns the output names this worker produced."""
    led = ExtractLedger(datadir)
    if init or not os.path.exists(led.path):
        led.files(init=True)
    names = sorted(os.listdir(videofolder))
    if shuffle_seed is not None:
        np.random.default_rng(shuffle_seed).shuffle(names)
    done = []
    for filename in names:
        if os.path.splitext(filename)[1] not in VIDEO_EXTENSIONS:
            continue
        outname = "video-%s-%s.pkl" % (filename[:3], mode)
        if led.claimed(outname):
            continue
        if not led.try_claim(outname):
            continue
        log(outname)
        led.add(outname)
        try:
            process_video(os.path.join(videofolder, filename), os.path.join(datadir, outname))
        finally:
            # finished: the ledger line (and the output file) keep the video closed.  Failed: the line stays, as in the
            # reference, until a run with init=True rebuilds the ledger from the files present -- and the claim must
            # not outlive this worker, or that run would skip the video forever.
            led.release(outname)
        done.append(outname)
    return done
