"""Every person on the batched estimators, tracked (extract.batch_every_person_extraction, BatchPoseEstimator
.every_person).  Prints one JSON line with
  - frames/s of the tracked video job on the device (decode, Batch_body, Batch_hand on both crops of every person,
    linking, file write) on a 720p MJPG clip, batch_size 32, two session pairs, one decode worker; and of the same job's
    host fallback on the same package estimators (batch_pose_mats_every_person + PersonLinker: crops cut with cv2,
    Batch_body and Batch_hand called on ToTensor-ed float batches); the two alternate and each figure is taken twice;
  - persons and crops per frame;
  - the hand half alone in crops/s on the decoded frames in pinned memory: wall clock of every_person on a batch minus
    that of Batch_body alone on the same batch (both end in a synchronise), against Batch_hand's 4286 crops/s
    (profiles/r02_batch_model.json);
  - the chunk-size sweep: the library rebuilt with kBatchEveryChunk = 16, 32 and 64 (api.cu recompiled, the other
    objects of the in-tree build reused, in a temporary directory), each measured in its own process on the same
    batches, the variants alternated and each taken twice.
The clip is one blurred-noise frame shifted by 3 pixels per frame, so the same persons recur; Kaiming body weights with
seed 62 assemble many persons with arms on it (as tools/bench_every_track.py).

    python tools/bench_batch_every_track.py [--out FILE]"""
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

H, W, FRAMES, BATCH, BLUR = 720, 1280, 128, 32, 2.25
CHUNKS = (16, 32, 64)
BATCH_HAND_CROPS_PER_SEC = 4286                              # profiles/r02_batch_model.json


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def write_clip(path):
    import cv2
    rng = np.random.default_rng(0)
    base = cv2.GaussianBlur(rng.integers(0, 256, (H, W + 3 * FRAMES, 3), dtype=np.uint8), (0, 0), BLUR)
    w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (W, H))
    for t in range(FRAMES):
        w.write(np.ascontiguousarray(base[:, 3 * (FRAMES - t):3 * (FRAMES - t) + W]))
    w.release()


def estimators():
    from oracle import openpose_oracle as O
    from pytorch_openpose_b200 import Batch_body, Batch_hand, BatchPoseEstimator
    body = Batch_body(O.make_weights("body", 62, "kaiming"))
    hand = Batch_hand(O.make_weights("hand", 5, "kaiming"))
    return body, hand, BatchPoseEstimator(body, hand)


def pinned_batches(clip):
    import torch
    from pytorch_openpose_b200 import extract
    return [torch.from_numpy(np.array(fr)).pin_memory() for fr, _ in extract.FrameBatches(clip, None, batch=BATCH)]


def device_resident(body, est, batches, reps=3):
    """(frames/s of every_person, hand-half crops/s, persons per frame) over `reps` passes over the batches"""
    pair = est.sessions(1)[0]
    t_all = t_body = 0.0
    persons = []
    for _ in range(reps):
        for b in batches:
            t0 = time.perf_counter()
            est.submit_every_person(b, pair, where=2)
            recs = est.collect_every_person(pair)
            t1 = time.perf_counter()
            body.submit_frames(b.numpy(), where=2)
            body.collect()
            t_all += t1 - t0
            t_body += time.perf_counter() - t1
            persons += [len(r) for r in recs]
    frames = reps * sum(len(b) for b in batches)
    return frames / t_all, 2 * sum(persons) / (t_all - t_body), persons


def build_variant(chunk, out_dir):
    from pytorch_openpose_b200 import build as B
    B.build()
    src = open(os.path.join(B.CSRC, "api.cu")).read()
    patched, n = re.subn(r"constexpr int kBatchEveryChunk = \d+;", "constexpr int kBatchEveryChunk = %d;" % chunk, src)
    assert n == 1
    cu, obj, so = (os.path.join(out_dir, "api_c%d.%s" % (chunk, ext)) for ext in ("cu", "o", "so"))
    with open(cu, "w") as f:
        f.write(patched)
    nvcc = B._nvcc()
    subprocess.run([nvcc] + B.ARCH + B.COMMON + ["-I", B.CSRC, "-c", cu, "-o", obj], check=True)
    objs = [os.path.join(B.BUILD, s.replace(".cu", ".o")) for s in B.SOURCES if s != "api.cu"]
    subprocess.run([nvcc] + B.ARCH + ["-shared", "-o", so] + objs + [obj, "-Xcompiler", "-fPIC", "-cudart", "static"],
                   check=True)
    return so


def sweep_worker(lib_path, clip):
    from pytorch_openpose_b200 import _lib
    _lib.LIB_PATH = lib_path
    body, _, est = estimators()
    batches = pinned_batches(clip)
    device_resident(body, est, batches, reps=1)                          # plans, tables, graphs
    fps, crops, _ = device_resident(body, est, batches)
    print(json.dumps({"frames_per_sec": round(fps, 2), "hand_crops_per_sec": round(crops, 1)}))


def main():
    from pytorch_openpose_b200 import extract
    info = gpu_info()
    tmp = tempfile.mkdtemp()
    clip = os.path.join(tmp, "clip.avi")
    write_clip(clip)
    body, hand, est = estimators()

    def device_job():
        t0 = time.perf_counter()
        out = extract.batch_every_person_extraction(clip, os.path.join(tmp, "d.pkl"), BATCH, None, body, hand,
                                                    log=lambda s: None, sessions=2)
        return time.perf_counter() - t0, out

    def host_job():
        t0 = time.perf_counter()
        out = extract.batch_every_person_extraction(clip, os.path.join(tmp, "h.pkl"), BATCH, None, lambda b: body(b),
                                                    lambda c: hand(c), log=lambda s: None)
        return time.perf_counter() - t0, out

    device_job()                                                         # plans, tables, graphs
    fps = {"device_job": [], "host_fallback_job": []}
    for _ in range(2):                                                   # alternated, twice: the spread
        for name, fn in (("device_job", device_job), ("host_fallback_job", host_job)):
            dt, out = fn()
            fps[name].append(round(FRAMES / dt, 2))
    tracks = out["tracks"]

    batches = pinned_batches(clip)
    device_resident(body, est, batches, reps=1)
    resident = [device_resident(body, est, batches) for _ in range(2)]
    persons = resident[0][2][:FRAMES]

    sweep = {c: [] for c in CHUNKS}
    libs = {c: build_variant(c, tmp) for c in CHUNKS}
    for _ in range(2):
        for c in CHUNKS:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--sweep-worker", libs[c], clip],
                               capture_output=True, text=True, cwd=ROOT)
            assert r.returncode == 0, r.stderr[-3000:]
            sweep[c].append(json.loads(r.stdout.strip().splitlines()[-1]))

    result = dict(info, metric="batch_every_person_tracked_frames_per_sec_720p", frames=FRAMES, batch=BATCH, blur=BLUR,
                  frames_per_sec=fps,
                  persons_per_frame_min_mean_max=[min(persons), round(float(np.mean(persons)), 1), max(persons)],
                  crops_per_frame_mean=round(2 * float(np.mean(persons)), 1),
                  tracks=len(tracks), longest_track_frames=max(len(m) for _, m in tracks),
                  device_resident_frames_per_sec=[round(r[0], 2) for r in resident],
                  hand_half_crops_per_sec=[round(r[1], 1) for r in resident],
                  batch_hand_crops_per_sec_reference=BATCH_HAND_CROPS_PER_SEC,
                  chunk_sweep={str(c): v for c, v in sweep.items()},
                  note="wall clock; jobs include decode (1 worker), the tracker and the file write; device-resident "
                       "figures on pinned decoded batches of 32 frames, hand half = every_person minus Batch_body alone "
                       "on the same batch; chunk sweep: one process per library variant, alternated")
    line = json.dumps(result)
    print(line)
    if "--out" in sys.argv:
        with open(sys.argv[sys.argv.index("--out") + 1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    if "--sweep-worker" in sys.argv:
        i = sys.argv.index("--sweep-worker")
        sweep_worker(sys.argv[i + 1], sys.argv[i + 2])
    else:
        main()
