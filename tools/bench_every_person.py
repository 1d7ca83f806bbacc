"""Every person of every frame (PoseEstimator.every_person, opb_pose_every_*) against the host loop it replaces: Body,
util.handDetect on every person and one Hand call per box (motion.pose_mats_every_person).  Prints one JSON line with
  - frames/s of both on the same 720p frames (pageable host memory, body and hand at 4 scales), the
    device path in batches of 8 frames; the two are alternated and each figure is taken twice;
  - persons and hand boxes per frame;
  - the hand half alone in crops/s: the device path's time per batch minus that of the body network alone on the same
    batch (Body.batch), over the boxes of the batch.
Random weights find nobody on most images.  Kaiming body weights with seed 62 assemble people with arms on blurred
noise; the blur width is the first of a fixed list that gives at least two hand boxes per frame, and is reported.
Every configuration is warmed up first; results of the two paths are checked to be identical.

    python tools/bench_every_person.py"""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2                                                               # noqa: E402
from oracle import openpose_oracle as O                                 # noqa: E402
from pytorch_openpose_b200 import Body, Hand, motion, util              # noqa: E402

H, W, BATCH, MIN_SECONDS = 720, 1280, 8, 3.0


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def frames_for(blur, n, seed=0):
    rng = np.random.default_rng(seed)
    return np.stack([cv2.GaussianBlur(rng.integers(0, 256, (H, W, 3), dtype=np.uint8), (0, 0), blur) for _ in range(n)])


body = Body(O.make_weights("body", 62, "kaiming"), scale_search=[0.5, 1.0, 1.5, 2.0])
hand = Hand(O.make_weights("hand", 5, "kaiming"))                       # default scale_search: 4 scales
est = motion.PoseEstimator(body, hand)
for blur in (3.0, 2.75, 2.5, 2.25, 2.0):
    frames = frames_for(blur, BATCH)
    boxes = [util.handDetect(*body(f), f) for f in frames]
    if sum(len(b) for b in boxes) >= 2 * BATCH:
        break
V = sum(len(b) for b in boxes)


def device(reps):
    t0 = time.perf_counter()
    for _ in range(reps):
        out = est.every_person(frames)
    return time.perf_counter() - t0, out


def host(reps):
    t0 = time.perf_counter()
    for _ in range(reps):
        out = [motion.pose_mats_every_person(f, body, hand) for f in frames]
    return time.perf_counter() - t0, out


def body_only(reps):
    t0 = time.perf_counter()
    for _ in range(reps):
        body.batch(frames)
    return time.perf_counter() - t0, None


for fn in (device, host, body_only):
    fn(3)                                                                # plans, tables, graphs
reps = {}
for name, fn in (("device", device), ("host", host), ("body_only", body_only)):
    dt, _ = fn(1)
    reps[name] = max(2, int(MIN_SECONDS / dt + 0.5))
fps = {"device": [], "host": []}
batch_s = {"device": [], "body_only": []}
for _ in range(2):                                                      # alternated, twice: the spread
    for name, fn in (("device", device), ("host", host), ("body_only", body_only)):
        dt, out = fn(reps[name])
        if name != "body_only":
            fps[name].append(round(reps[name] * BATCH / dt, 2))
            if name == "device":
                dev_out = out
            else:
                assert all(np.array_equal(a, b) for a, b in zip(dev_out, out)), "device and host records differ"
        if name != "host":
            batch_s[name].append(dt / reps[name])
crops = [round(V / (d - b), 1) for d, b in zip(batch_s["device"], batch_s["body_only"])]
persons = [len(r) for r in dev_out]
print(json.dumps(dict(gpu_info(), metric="every_person_frames_per_sec_720p", frames_per_sec=fps,
                      hand_half_crops_per_sec=crops, batch=BATCH, blur=blur, persons_per_frame=persons,
                      hand_boxes_per_frame=[len(b) for b in boxes],
                      hands_with_key_points=int(sum(int((r[:, 18:39, 2] > 0).any(axis=1).sum() +
                                                        (r[:, 39:, 2] > 0).any(axis=1).sum()) for r in dev_out)),
                      body_scales=body.scale_search, hand_scales=hand.scale_search, repetitions=reps,
                      note="wall clock, frames in pageable host memory, results on the host; device path in batches "
                           "of %d frames, host path frame by frame; crops/s = hand boxes of the batch over the device "
                           "path's batch time minus Body.batch's; each figure measured twice, alternated" % BATCH)))
