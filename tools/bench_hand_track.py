"""The batched hand job (Batch_hand_extraction, srcmx/Batch_motion_Estimation.py:19-63) on the device.  Prints one JSON
line with
  (a) frames/s of Batch_hand.track's device pipeline on device-resident 720p frames, 32 frames per batch, 2 and 3
      sessions in flight (pose -> boxes -> crops -> Batch_hand -> HandMat), timed with CUDA events after warm-up;
  (b) frames/s of the whole job `extract.batch_hand_extraction` on a seeded 720p MJPG file (wall clock: decode, crops,
      network, file write): the host path (OPB_HOST_HANDS=1) against the device path with 1 and 4 decode workers.
Every frame has a synthetic pose with two valid hand boxes (~150-200 px, a new size every frame), so both hands really
go through the network.  Random-init hand weights (no checkpoints offline).

    python tools/bench_hand_track.py [frames_of_the_video=256]"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2                                                     # noqa: E402
import torch                                                   # noqa: E402
from pytorch_openpose_b200 import Batch_hand, extract          # noqa: E402
from pytorch_openpose_b200.model import random_checkpoint      # noqa: E402

H, W, B = 720, 1280, 32


def pose_track(n):
    mats = np.zeros((n, 18, 3))
    for k in range(n):
        joints = {1: (640, 200), 2: (500, 200), 3: (430 + k % 17, 330), 4: (380 + 2 * (k % 13), 460 + k % 19),
                  5: (780, 200), 6: (850 - k % 16, 330), 7: (900 - 2 * (k % 11), 460 + k % 23)}
        for j, (x, y) in joints.items():
            mats[k, j] = (x, y, 0.9)
    return mats


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


est = Batch_hand(random_checkpoint("hand", 0))
rng = np.random.default_rng(0)
base = np.stack([cv2.GaussianBlur(rng.integers(0, 256, (H, W, 3), dtype=np.uint8), (0, 0), 5) for _ in range(B)])
frames_dev = torch.from_numpy(base).cuda()
poses = pose_track(B)


def resident(n_sessions, iters=60):
    ss = extract._job_sessions(est, n_sessions)

    def run(k):
        for it in range(k):
            s = ss[it % n_sessions]
            if it >= n_sessions:
                est.collect_track(s)
            est.submit_track(frames_dev, poses, s)
        for it in range(max(0, k - n_sessions), k):
            est.collect_track(ss[it % n_sessions])

    run(4 * n_sessions)                                        # plans, tables, graphs
    ss[0].mark(0)
    run(iters)
    for s in ss:
        s.mark(1)
    ms = max(ss[0].elapsed_ms(0, s, 1) for s in ss)
    return round(iters * B / (ms / 1e3), 1)


a = {str(k): resident(k) for k in (2, 3)}
mats = est.track(base, poses)
both = int(((mats[:, :21, 2] > 0).any(1) & (mats[:, 21:, 2] > 0).any(1)).sum())

N = int(sys.argv[1]) if len(sys.argv) > 1 else 256
d = tempfile.mkdtemp()
path = os.path.join(d, "v.avi")
wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (W, H))
for i in range(N):
    wr.write(np.roll(base[i % 8], 7 * i, axis=1))
wr.release()
track = pose_track(N)


def job(workers, host):
    if host:
        os.environ["OPB_HOST_HANDS"] = "1"
    try:
        kw = {} if host else {"decode_workers": workers, "sessions": 3}
        extract.batch_hand_extraction(path, track, None, os.path.join(d, "w.pkl"), est, batchsize=B, log=lambda m: None, **kw)
        t0 = time.perf_counter()
        mat = extract.batch_hand_extraction(path, track, None, os.path.join(d, "o.pkl"), est, batchsize=B,
                                            log=lambda m: None, **kw)
        return round(len(mat) / (time.perf_counter() - t0), 1), mat
    finally:
        os.environ.pop("OPB_HOST_HANDS", None)


host_fps, host_mat = job(1, True)
b = {"host_path_1_worker": host_fps}
for k in (1, 4):
    b["device_path_%d_workers" % k], dev_mat = job(k, False)
# the two paths on the same file: the host crops go through IPP's resize here (1 LSB on some pixels), so the key points
# may differ slightly; the bit-exact comparison with IPP off is tests/test_gpu_hand_track.py
b["max_abs_diff_device_vs_host"] = float(np.abs(dev_mat - host_mat).max())
print(json.dumps(dict(gpu_info(), metric="hand_track_frames_per_sec_720p",
                      device_resident_fps_by_sessions=a, frames_with_both_hands=both, frames_per_batch=B,
                      job_fps=b, video_frames=N, host_cores=os.cpu_count(),
                      note="(a) CUDA events on the sessions' streams over 60 batches after warm-up; (b) wall clock of the "
                           "whole job incl. MJPG decode and the file write")))
