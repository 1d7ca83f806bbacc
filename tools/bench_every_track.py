"""Person tracks on the device (extract_every_person_from_video, opb_pose_every_wait_tracked) against what they add to.
Prints one JSON line with
  - frames/s of the tracked video job (decode, body and hands of every person, linking, file write) on a 720p MJPG
    file, and of the untracked every-person batches on the same decoded frames (same decode loop, two session pairs in
    flight, no linking, no file); the two are alternated and each figure is taken twice;
  - the link launch's own device time per batch of 8 frames: CUDA events recorded on the session's stream right before
    and after it (session profiling, the "track_link" mark);
  - host linking (motion.PersonLinker) on the same records, per batch of 8 frames.
The clip is one blurred-noise frame shifted by 3 pixels per frame, so the same persons recur; Kaiming body weights with
seed 62 assemble people with arms on it (as in tools/bench_every_person.py).

    python tools/bench_every_track.py [--out FILE]"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2                                                               # noqa: E402
from oracle import openpose_oracle as O                                 # noqa: E402
from pytorch_openpose_b200 import Body, Hand, extract, motion           # noqa: E402

H, W, FRAMES, BATCH, BLUR = 720, 1280, 64, 8, 2.25
GATE = dict(max_gap=15, max_dist=0.1 * H, min_joints=3)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def write_clip(path):
    rng = np.random.default_rng(0)
    base = cv2.GaussianBlur(rng.integers(0, 256, (H, W + 3 * FRAMES, 3), dtype=np.uint8), (0, 0), BLUR)
    w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (W, H))
    for t in range(FRAMES):
        w.write(np.ascontiguousarray(base[:, 3 * (FRAMES - t):3 * (FRAMES - t) + W]))
    w.release()


body = Body(O.make_weights("body", 62, "kaiming"), scale_search=[0.5, 1.0, 1.5, 2.0])
hand = Hand(O.make_weights("hand", 5, "kaiming"))
est = motion.PoseEstimator(body, hand)
tmp = tempfile.mkdtemp()
clip, outpath = os.path.join(tmp, "clip.avi"), os.path.join(tmp, "tracks.pkl")
write_clip(clip)


def tracked():
    t0 = time.perf_counter()
    out = extract.extract_every_person_from_video(clip, outpath, None, body, hand, batch=BATCH, sessions=2,
                                                  log=lambda s: None, **GATE)
    return time.perf_counter() - t0, out


def untracked():
    pairs = est.sessions(2)
    t0 = time.perf_counter()
    pending, recs = [], []
    for frames, first, nv in extract.FrameBatches(clip, None, batch=BATCH, depth=5, pinned=True, pad_last=True,
                                                  ordered=True):
        if len(pending) == 2:
            recs += est.collect_every_person(pending.pop(0))
        pair = next(c for c in pairs if c not in pending)
        est.submit_every_person(frames, pair, where=2)
        pending.append(pair)
    while pending:
        recs += est.collect_every_person(pending.pop(0))
    return time.perf_counter() - t0, recs


for fn in (tracked, untracked):
    fn()                                                                 # plans, tables, graphs
fps = {"tracked_job": [], "untracked_batches": []}
for _ in range(2):                                                      # alternated, twice: the spread
    for name, fn in (("tracked_job", tracked), ("untracked_batches", untracked)):
        dt, out = fn()
        fps[name].append(round(FRAMES / dt, 2))
        if name == "tracked_job":
            tracks = out["tracks"]
        else:
            records = out

# the link launch alone: profiling on one session pair, one batch at a time
batches = [np.array(fr) for fr, _, _ in extract.FrameBatches(clip, None, batch=BATCH, pad_last=True)]
bs, hs = est.sessions(1)[0]
tr = est.tracker(**GATE)
link_ms = []
for b in batches:
    bs.set_profiling(True)
    est.submit_every_person(b, (bs, hs))
    est.collect_every_person((bs, hs), tracker=tr)
    marks = dict((name, ms) for name, ms, _ in bs.profile())
    link_ms.append(round(marks["track_link"], 4))
bs.set_profiling(False)

# host linking on the same records
lk = motion.PersonLinker(**GATE)
host_ms = []
for i in range(0, FRAMES, BATCH):
    t0 = time.perf_counter()
    for r in records[i:i + BATCH]:
        lk.link(r)
    host_ms.append(round(1000 * (time.perf_counter() - t0), 3))

persons = [len(r) for r in records]
result = dict(gpu_info(), metric="every_person_tracked_frames_per_sec_720p", frames_per_sec=fps, frames=FRAMES,
              batch=BATCH, blur=BLUR, persons_per_frame_min_mean_max=[min(persons), round(float(np.mean(persons)), 1),
                                                                     max(persons)],
              tracks=len(tracks), longest_track_frames=max(len(m) for _, m in tracks),
              link_ms_per_batch_device=link_ms, link_ms_per_batch_device_median=float(np.median(link_ms)),
              link_ms_per_batch_host=host_ms, link_ms_per_batch_host_median=float(np.median(host_ms)),
              gate=GATE, body_scales=body.scale_search, hand_scales=hand.scale_search,
              note="wall clock for the job and the untracked batches (decode included, frames pinned, two session "
                   "pairs); link time from CUDA events around the link launch on the session stream (profiling on, "
                   "eager launches); host linking timed with perf_counter on the records of the untracked run")
line = json.dumps(result)
print(line)
if "--out" in sys.argv:
    with open(sys.argv[sys.argv.index("--out") + 1], "w") as f:
        f.write(line + "\n")
