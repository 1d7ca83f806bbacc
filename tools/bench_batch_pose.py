"""The one-pass body + hand job (BatchPoseEstimator / extract.batch_bodyhand_extraction) against the two-pass job it
replaces (Batch_body_extraction, then Batch_hand_extraction on its track; srcmx/Batch_motion_Estimation.py:19-112).
Prints one JSON line with
  (a) frames/s on 720p frames already in device memory, 16 and 32 frames per batch, 2 and 3 (body, hand) session pairs
      in flight: the one-pass sequence against the two separate device calls on the same frames -- Batch_body on the
      frames with body_pose on the fetched results for every batch, then Batch_hand's hand-track call on the frames and
      that track (wall clock; every run ends with its results on the host);
  (b) wall-clock frames/s of the whole job on a seeded 256-frame 720p MJPG file (decode, device work, both file
      writes) with 1 and 4 decode workers: batch_bodyhand_extraction against batch_body_extraction followed by
      batch_hand_extraction.
Random-init weights (no checkpoints offline) find nobody, so every hand box is missing; the hand network still runs on
all 2n crops of a batch (grey ones), so the device work per frame is that of real video.  Every configuration is warmed
up first, timed over several seconds of work, and measured twice to show the spread.

    python tools/bench_batch_pose.py [frames_of_the_video=256]"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2                                                               # noqa: E402
import torch                                                             # noqa: E402
from pytorch_openpose_b200 import Batch_body, Batch_hand, BatchPoseEstimator, _lib, extract      # noqa: E402
from pytorch_openpose_b200.model import random_checkpoint                # noqa: E402

H, W = 720, 1280
FRAMES_PER_RUN = 4096                                                    # ~2-4 s of device work per measurement


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


body = Batch_body(random_checkpoint("body", 0))
hand = Batch_hand(random_checkpoint("hand", 0))
est = BatchPoseEstimator(body, hand)
rng = np.random.default_rng(0)
base = np.stack([cv2.GaussianBlur(rng.integers(0, 256, (H, W, 3), dtype=np.uint8), (0, 0), 5) for _ in range(32)])
frames_dev = torch.from_numpy(base).cuda()
body_s = extract._job_sessions(body, 3)
hand_s = extract._job_sessions(hand, 3)


def one_pass(B, P, iters):
    pairs = est.sessions(P)
    x = frames_dev[:B]
    t0 = time.perf_counter()
    for it in range(iters):
        if it >= P:
            est.collect(pairs[it % P])
        est.submit(x, pairs[it % P])
    out = [est.collect(pairs[it % P]) for it in range(max(0, iters - P), iters)]
    return time.perf_counter() - t0, out[-1]


def two_pass(B, P, iters):
    """The two jobs' device calls on the same frames: all body batches (results fetched, body_pose per frame), then all
    hand-track batches on that track."""
    x = frames_dev[:B]
    L = _lib.lib()
    t0 = time.perf_counter()
    motion = [None] * iters

    def body_retire(it):
        motion[it] = np.stack([extract.body_pose(c, s)[0] for c, s in body.collect(body_s[it % P])])

    for it in range(iters):
        if it >= P:
            body_retire(it - P)
        s = body_s[it % P]
        s._batch, s._shape, s._keepalive = B, (B, H, W), x
        _lib.check(L.opb_batch_body_submit_u8(s.handle, x.data_ptr(), 1, B, H, W, float(body.scale_search)))
    for it in range(max(0, iters - P), iters):
        body_retire(it)
    hands = None
    for it in range(iters):
        if it >= P:
            hand.collect_track(hand_s[it % P])
        hand.submit_track(x, motion[it], hand_s[it % P])
    for it in range(max(0, iters - P), iters):
        hands = hand.collect_track(hand_s[it % P])
    return time.perf_counter() - t0, (motion[-1], hands)


a = {}
for B in (16, 32):
    iters = FRAMES_PER_RUN // B
    for P in (2, 3):
        for fn in (one_pass, two_pass):
            fn(B, P, 4 * P)                                              # plans, tables, graphs
        runs = {"one_pass": [], "two_pass": []}
        for _ in range(2):                                              # alternated, twice: the spread
            for name, fn in (("one_pass", one_pass), ("two_pass", two_pass)):
                dt, res = fn(B, P, iters)
                runs[name].append(round(iters * B / dt, 1))
                if name == "one_pass":
                    one_res = res
                else:
                    assert np.array_equal(one_res[0], res[0]) and np.array_equal(one_res[1], res[1])
        a["%d_frames_%d_pairs" % (B, P)] = runs

N = int(sys.argv[1]) if len(sys.argv) > 1 else 256
d = tempfile.mkdtemp()
path = os.path.join(d, "v.avi")
wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (W, H))
for i in range(N):
    wr.write(np.roll(base[i % 8], 7 * i, axis=1))
wr.release()
quiet = lambda m: None                                                  # noqa: E731


def job_one(workers):
    return extract.batch_bodyhand_extraction(path, os.path.join(d, "b1.pkl"), os.path.join(d, "h1.pkl"), 32, None, body,
                                             hand, log=quiet, decode_workers=workers, sessions=3)


def job_two(workers):
    m = extract.batch_body_extraction(path, os.path.join(d, "b2.pkl"), 32, None, body, log=quiet,
                                      decode_workers=workers, sessions=3)
    return m, extract.batch_hand_extraction(path, m, None, os.path.join(d, "h2.pkl"), hand, batchsize=32, log=quiet,
                                            decode_workers=workers, sessions=3)


b = {}
for k in (1, 4):
    for fn in (job_one, job_two):
        fn(k)                                                           # warm-up
    runs = {"one_pass": [], "two_pass": []}
    for _ in range(2):
        for name, fn in (("one_pass", job_one), ("two_pass", job_two)):
            t0 = time.perf_counter()
            m, h = fn(k)
            runs[name].append(round(len(m) / (time.perf_counter() - t0), 1))
    b["%d_decode_workers" % k] = runs
import joblib                                                           # noqa: E402
same = all(np.array_equal(joblib.load(os.path.join(d, x + "1.pkl")), joblib.load(os.path.join(d, x + "2.pkl")))
           for x in ("b", "h"))
print(json.dumps(dict(gpu_info(), metric="bodyhand_frames_per_sec_720p", device_resident_fps=a, job_fps=b,
                      job_files_identical=same, video_frames=N, host_cores=os.cpu_count(),
                      note="(a) wall clock, %d frames per run after warm-up, frames in device memory; (b) wall clock of "
                           "the whole job incl. MJPG decode and both file writes, 32 frames per batch, 3 session "
                           "pairs; each figure measured twice, one-pass and two-pass alternated" % FRAMES_PER_RUN)))
