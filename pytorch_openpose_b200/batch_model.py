"""`Batch_body(model_path)(batch_images)` / `Batch_hand(model_path)(batch_imgs)` -- drop-ins for the reference's batched
estimators (srcmx/Batch_model.py:107-406, SURVEY.md 8f row N2) on libopenpose_b200.so.

Same call contract as the reference: `batch_images` is a float (B, 3, h, w) tensor/array in [0, 1] (what
`transforms.ToTensor()` gives); Batch_body returns `[(candidates, subset)] * B`, Batch_hand an array (B, 21, 3).
The numerics differ from `Body` / `Hand` on purpose, exactly as in the reference: torch-bicubic float resizes, one
scale (0.5), a 5x5 blur instead of the sigma-3 Gaussian, peaks found AND scored on the blurred map, hand threshold
0.035."""
import ctypes

import numpy as np

from . import _lib
from .body import _load_checkpoint


def _as_frames_u8(frames, where):
    """Decoded frames (B, h, w, 3) uint8 as they come out of cv2 -> (pointer, keepalive, (B, h, w))."""
    arr = np.ascontiguousarray(frames, dtype=np.uint8)
    if arr.ndim != 4 or arr.shape[3] != 3:
        raise ValueError("expected (B, h, w, 3) uint8 frames")
    return arr.ctypes.data, arr, arr.shape[:3]


def _as_track_frames(frames, where):
    """-> (pointer, where, keepalive, (B, h, w)) of (B, h, w, 3) uint8 frames: torch CUDA tensors are read in place
    (where=1), pinned CPU tensors straight from their pages (where=2); anything else as `where` says."""
    if hasattr(frames, "detach"):
        import torch
        t = frames.detach()
        if t.is_cuda or t.is_pinned():
            if t.dtype != torch.uint8 or t.dim() != 4 or t.shape[3] != 3:
                raise ValueError("expected (B, h, w, 3) uint8 frames")
            t = t.contiguous()
            if t.is_cuda:
                torch.cuda.current_stream(t.device).synchronize()       # producer work is on torch's stream
            return t.data_ptr(), (1 if t.is_cuda else 2), t, tuple(t.shape[:3])
        frames = t.numpy()
    ptr, keep, shape = _as_frames_u8(frames, where)
    return ptr, where, keep, shape


def _as_float_batch(batch):
    """-> (pointer, where, keepalive, shape).  torch CUDA tensors are read in place (where=1), pinned CPU tensors are
    copied straight from their pages (where=2); anything else goes through the library's pinned staging buffer."""
    if hasattr(batch, "detach"):
        t = batch.detach()
        if t.dim() != 4 or t.shape[1] != 3:
            raise ValueError("expected a (B, 3, h, w) float batch")
        import torch
        if t.is_cuda or t.is_pinned():
            t = t.to(torch.float32).contiguous()
            if t.is_cuda:
                torch.cuda.current_stream(t.device).synchronize()       # producer work is on torch's stream
            return t.data_ptr(), (1 if t.is_cuda else 2), t, tuple(t.shape)
        batch = t.numpy()
    arr = np.ascontiguousarray(batch, dtype=np.float32)
    if arr.ndim != 4 or arr.shape[1] != 3:
        raise ValueError("expected a (B, 3, h, w) float batch")
    return arr.ctypes.data, 0, arr, arr.shape


class Batch_body(object):
    MAX_BATCH = 16

    def __init__(self, model_path, device=None):
        weights = model_path if isinstance(model_path, dict) else _load_checkpoint(model_path)
        self.net = _lib.Net(_lib.NET_BODY, weights, device)
        self._session = self.net.session()
        self.scale_search = 0.5                        # srcmx/Batch_model.py:118

    def submit(self, batch_images, session=None):
        s = session or self._session
        ptr, where, s._keepalive, (B, _, h, w) = _as_float_batch(batch_images)
        s._batch, s._shape = B, (B, h, w)
        _lib.check(_lib.lib().opb_batch_body_submit(s.handle, ptr, where, B, h, w, float(self.scale_search)))

    def submit_frames(self, frames_u8, session=None, where=0):
        """Same as `submit(ToTensor(frames))` for decoded (B, h, w, 3) uint8 frames, without the host-side float
        conversion: the division by 255 happens on the device (bit-identical).  where=2: `frames_u8` is pinned."""
        s = session or self._session
        ptr, s._keepalive, (B, h, w) = _as_frames_u8(frames_u8, where)
        s._batch, s._shape = B, (B, h, w)
        _lib.check(_lib.lib().opb_batch_body_submit_u8(s.handle, ptr, where, B, h, w, float(self.scale_search)))

    def collect(self, session=None):
        s = session or self._session
        L = _lib.lib()
        n = s._batch
        nc, ns, st = (ctypes.c_int * n)(), (ctypes.c_int * n)(), (ctypes.c_int * n)()
        _lib.check(L.opb_body_wait_batch(s.handle, nc, ns, st))
        out = []
        for f in range(n):
            candidate = np.empty((nc[f], 4), dtype=np.float64)
            subset = np.empty((ns[f], 20), dtype=np.float64)
            _lib.check(L.opb_body_fetch_frame(s.handle, f, candidate.ctypes.data, nc[f], subset.ctypes.data, ns[f]))
            out.append((np.array([]) if nc[f] == 0 else candidate, subset))
        return out

    def __call__(self, batch_images):
        results = []
        for lo in range(0, len(batch_images), self.MAX_BATCH):          # activations of 16 frames per launch set
            self.submit(batch_images[lo:lo + self.MAX_BATCH])
            results.extend(self.collect())
        return results

    def last_maps(self, session=None):
        """(blurred heat (B,h,w,19), paf (B,h,w,38)) float32 of the last submitted chunk (Batch_model.py:182-183)."""
        s = session or self._session
        B, h, w = s._shape
        blurred = np.empty((B, 19, h, w), dtype=np.float32)
        paf = np.empty((B, 38, h, w), dtype=np.float32)
        _lib.check(_lib.lib().opb_batch_maps(s.handle, blurred.ctypes.data))
        _lib.check(_lib.lib().opb_body_maps(s.handle, None, paf.ctypes.data))
        return np.ascontiguousarray(blurred.transpose(0, 2, 3, 1)), np.ascontiguousarray(paf.transpose(0, 2, 3, 1))


class Batch_hand(object):
    MAX_BATCH = 64

    def __init__(self, model_path, device=None):
        weights = model_path if isinstance(model_path, dict) else _load_checkpoint(model_path)
        self.net = _lib.Net(_lib.NET_HAND, weights, device)
        self._session = self.net.session()

    def submit(self, batch_imgs, session=None):
        s = session or self._session
        ptr, where, s._keepalive, (B, _, h, w) = _as_float_batch(batch_imgs)
        s._n, s._shape = B, (B, h, w)
        if h % 8 or w % 8:
            raise ValueError("Batch_hand crops must have sides that are multiples of 8: the reference upsamples the "
                             "stride-8 maps by exactly 8 (srcmx/Batch_model.py:377)")
        _lib.check(_lib.lib().opb_batch_hand_submit(s.handle, ptr, where, B, h, w))

    def submit_frames(self, crops_u8, session=None, where=0):
        """`submit(ToTensor(crops))` for (B, h, w, 3) uint8 crops; /255 on the device."""
        s = session or self._session
        ptr, s._keepalive, (B, h, w) = _as_frames_u8(crops_u8, where)
        s._n, s._shape = B, (B, h, w)
        if h % 8 or w % 8:
            raise ValueError("Batch_hand crops must have sides that are multiples of 8 (srcmx/Batch_model.py:377)")
        _lib.check(_lib.lib().opb_batch_hand_submit_u8(s.handle, ptr, where, B, h, w))

    def collect(self, session=None):
        s = session or self._session
        peaks = np.empty((s._n, 21, 3), dtype=np.float64)
        _lib.check(_lib.lib().opb_hand_wait(s.handle, peaks.ctypes.data))
        return peaks

    TRACK_BATCH = MAX_BATCH // 2                      # frames per track submit: two crops each

    def submit_track(self, frames_u8, poses, session=None, where=0, boxsize=368):
        """One batch of `Batch_hand_extraction` (srcmx/Batch_motion_Estimation.py:19-63) on the device: ROI-cropped
        (B, h, w, 3) uint8 frames and their saved (B, 18, 3) body poses -> both hand crops of every frame
        (`extract.hand_crops_from_pose`), Batch_hand on them and the key points back in ROI coordinates
        (`collect_track`).  where: 0 pageable, 1 device (a CUDA tensor is always read in place), 2 pinned."""
        s = session or self._session
        ptr, where, keep, (B, h, w) = _as_track_frames(frames_u8, where)
        p = np.ascontiguousarray(poses, dtype=np.float64)
        if p.shape != (B, 18, 3):
            raise ValueError("expected (%d, 18, 3) poses for %d frames, got %s" % (B, B, p.shape))
        if boxsize % 8:
            raise ValueError("boxsize must be a multiple of 8 (srcmx/Batch_model.py:377)")
        s._keepalive, s._track_n, s._track_box = (keep, p), B, int(boxsize)
        _lib.check(_lib.lib().opb_hand_track_submit(s.handle, ptr, where, B, h, w, p.ctypes.data, int(boxsize)))

    def collect_track(self, session=None):
        """HandMat (B, 42, 3) float64 of the last `submit_track`: rows 0-20 left hand, 21-41 right hand."""
        s = session or self._session
        mats = np.empty((s._track_n, 42, 3), dtype=np.float64)
        _lib.check(_lib.lib().opb_hand_track_wait(s.handle, mats.ctypes.data))
        return mats

    def track_crops(self, session=None):
        """The (2B, boxsize, boxsize, 3) uint8 crops of the last `submit_track` (slot 2f: left hand of frame f)."""
        s = session or self._session
        crops = np.empty((2 * s._track_n, s._track_box, s._track_box, 3), dtype=np.uint8)
        _lib.check(_lib.lib().opb_hand_track_crops(s.handle, crops.ctypes.data))
        return crops

    def track(self, frames, poses, boxsize=368):
        """HandMat (B, 42, 3) of `Batch_hand_extraction` for frames (B, h, w, 3) uint8 and poses (B, 18, 3)."""
        out = []
        for lo in range(0, len(frames), self.TRACK_BATCH):
            self.submit_track(frames[lo:lo + self.TRACK_BATCH], poses[lo:lo + self.TRACK_BATCH], boxsize=boxsize)
            out.append(self.collect_track())
        return np.concatenate(out, 0)

    def __call__(self, batch_imgs):
        out = []
        for lo in range(0, len(batch_imgs), self.MAX_BATCH):
            self.submit(batch_imgs[lo:lo + self.MAX_BATCH])
            out.append(self.collect())
        return np.concatenate(out, 0)

    def last_maps(self, session=None):
        """blurred heat maps (B,h,w,22) float32 of the last submitted chunk (Batch_model.py:378-385)."""
        s = session or self._session
        B, h, w = s._shape
        blurred = np.empty((B, 22, h, w), dtype=np.float32)
        _lib.check(_lib.lib().opb_batch_maps(s.handle, blurred.ctypes.data))
        return np.ascontiguousarray(blurred.transpose(0, 2, 3, 1))


class BatchPoseEstimator(object):
    """`Batch_body_extraction` followed by `Batch_hand_extraction` (srcmx/Batch_motion_Estimation.py:19-112) for batches
    of ROI-cropped frames in one device pass -- the batched counterpart of `motion.PoseEstimator`.  The frames go up
    once; Batch_body, the person with the largest left-shoulder x, both hand boxes from its body rows (as
    HandImageDataset derives them from the saved MotionMat), both crops cut from the frames in device memory, Batch_hand
    on all of them and the key points in ROI coordinates all run as one launch sequence.  Only the two tracks come back,
    equal to what the two jobs write: MotionMat (n, 18, 3) and HandMat (n, 42, 3).

    `batch_body` / `batch_hand`: this package's `Batch_body` / `Batch_hand` (their scale_search, 0.5, is used).  A hand
    box of width 0, on which the reference's cv2.resize raises, counts as a missing hand (as in `Batch_hand.track`).

    `every_person` / `submit_every_person` / `collect_every_person` run the same sequence for every person of every
    frame (`extract.batch_pose_mats_every_person` states the contract); `tracker` links them across batches."""

    MAX_BATCH = 32                                    # frames per submit: 64 hand crops, like Batch_hand.TRACK_BATCH

    def __init__(self, batch_body, batch_hand):
        self.body, self.hand = batch_body, batch_hand

    def sessions(self, k):
        """k (body session, hand session) pairs kept on the estimator (plans and buffers are expensive to warm up)."""
        have = self.__dict__.setdefault("_session_pairs", [])
        while len(have) < k:
            have.append((self.body.net.session(), self.hand.net.session()))
        return have[:k]

    def submit(self, frames_u8, pair=None, where=0, boxsize=368):
        """Enqueue one batch of (B, h, w, 3) uint8 frames (numpy, or a pinned / CUDA torch tensor read in place).
        where: 0 pageable, 1 device, 2 pinned."""
        bs, hs = pair or self.sessions(1)[0]
        ptr, where, keep, (B, h, w) = _as_track_frames(frames_u8, where)
        bs._keepalive, bs._batch = keep, B
        _lib.check(_lib.lib().opb_batch_pose_submit(bs.handle, hs.handle, ptr, where, B, h, w,
                                                    float(self.body.scale_search), int(boxsize)))

    def collect(self, pair=None):
        """-> (MotionMat (B, 18, 3), HandMat (B, 42, 3)) float64 of the last `submit` on `pair`.  Raises IndexError
        where the reference's Batch_body would (src/body.py:173)."""
        bs, hs = pair or self.sessions(1)[0]
        motion = np.empty((bs._batch, 18, 3), dtype=np.float64)
        hand = np.empty((bs._batch, 42, 3), dtype=np.float64)
        status = (ctypes.c_int * bs._batch)()
        _lib.check(_lib.lib().opb_batch_pose_wait(bs.handle, motion.ctypes.data, hand.ctypes.data, status))
        return motion, hand

    def __call__(self, frames, boxsize=368):
        motion, hand = [], []
        for lo in range(0, len(frames), self.MAX_BATCH):
            self.submit(frames[lo:lo + self.MAX_BATCH], boxsize=boxsize)
            m, h = self.collect()
            motion.append(m)
            hand.append(h)
        return np.concatenate(motion, 0), np.concatenate(hand, 0)

    def submit_every_person(self, frames, pair=None, where=0, boxsize=368):
        """Every person of every frame: frames as for `submit`.  Batch_body, the body rows of every subset row, both
        hand crops of every person cut from the frames in device memory, Batch_hand on them in fixed chunks."""
        bs, hs = pair or self.sessions(1)[0]
        ptr, where, keep, (B, h, w) = _as_track_frames(frames, where)
        bs._keepalive, bs._batch = keep, B
        _lib.check(_lib.lib().opb_batch_pose_every_submit(bs.handle, hs.handle, ptr, where, B, h, w,
                                                          float(self.body.scale_search), int(boxsize)))

    def collect_every_person(self, pair=None, tracker=None, n_link=None):
        """-> list of B arrays (P_f, 60, 3) float64, equal to `extract.batch_pose_mats_every_person` frame by frame:
        record p of frame f is the [MotionMat | HandMat] row `collect` would return had its selection picked subset row
        p.  Raises IndexError where the reference's Batch_body would (src/body.py:173).

        With a `tracker` (`self.tracker(...)`): (records, ids), linked as `motion.PoseEstimator.collect_every_person`
        links them (the first `n_link` frames, default all; -1 for the others; a batch that raises is not linked)."""
        bs, hs = pair or self.sessions(1)[0]
        persons = (ctypes.c_int * bs._batch)()
        status = (ctypes.c_int * bs._batch)()
        L = _lib.lib()
        if tracker is None:
            _lib.check(L.opb_pose_every_wait(bs.handle, persons, status))
        else:
            n_link = bs._batch if n_link is None else int(n_link)
            _lib.check(L.opb_pose_every_wait_tracked(bs.handle, tracker.handle, n_link, persons, status))
        counts = list(persons)
        records = np.empty((sum(counts), 60, 3), dtype=np.float64)
        _lib.check(L.opb_pose_every_fetch(bs.handle, records.ctypes.data, len(records)))
        split = np.cumsum(counts)[:-1]
        if tracker is None:
            return np.split(records, split)
        ids = np.empty(len(records), dtype=np.int32)
        _lib.check(L.opb_pose_every_fetch_ids(bs.handle, ids.ctypes.data, len(ids)))
        return np.split(records, split), np.split(ids.astype(np.int64), split)

    def every_person(self, frames, tracker=None, boxsize=368):
        """One frame (h, w, 3) -> (P, 60, 3); a batch (B, h, w, 3) of at most MAX_BATCH frames -> list of B such
        arrays.  With a `tracker`: (records, ids) of the same shapes."""
        frames = frames if hasattr(frames, "shape") else np.asarray(frames)
        single = len(frames.shape) == 3
        self.submit_every_person(frames[None] if single else frames, boxsize=boxsize)
        out = self.collect_every_person(tracker=tracker)
        if tracker is None:
            return out[0] if single else out
        return (out[0][0], out[1][0]) if single else out

    def tracker(self, max_gap, max_dist, min_joints=3):
        """A device tracker for one video (`motion.PersonLinker`'s rule and arguments) on this estimator's GPU, for
        `collect_every_person(..., tracker=)`.  It keeps its tracks until `reset()`."""
        return _lib.Tracker(self.body.net.ctx, max_gap, max_dist, min_joints)
