"""MJPG decoding on the device against cv2.VideoCapture, alone and inside the batched extraction jobs.

    python tools/bench_decode.py [--frames 256] [--out profiles/r09_device_decode.json]

Two 720p MJPG clips (blurred noise, sigma 2 = high detail, sigma 8 = low detail) are written to a temporary directory.
Every figure is taken twice, the two sides alternating:
  * decode alone, frames/s: jpeg.DeviceFrames on two sessions in flight (batches of 32) against FrameBatches
    (cv2.VideoCapture) with 1 and 4 threads;
  * batch_body_extraction and batch_bodyhand_extraction, frames/s, decode="device" against decode_workers=4;
  * the entropy-decode kernel's share of the device decode time (torch.profiler, a run of its own).
The card's name and power limit are read in the same run."""
import argparse
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

from oracle import openpose_oracle as O                        # noqa: E402
from pytorch_openpose_b200 import extract, jpeg                 # noqa: E402
from pytorch_openpose_b200.batch_model import Batch_body, Batch_hand   # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except Exception as e:                                       # pragma: no cover
        return "unknown (%s)" % e


def picture(h, w, seed, sigma):
    import cv2
    return cv2.GaussianBlur(np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), sigma)


def packet_sizes(path):
    import cv2
    cap = cv2.VideoCapture(path)
    cap.set(cv2.CAP_PROP_FORMAT, -1)
    sizes = []
    while True:
        ok, p = cap.read()
        if not ok:
            break
        sizes.append(p.size)
    cap.release()
    return sizes


def write_clip(path, n, sigma):
    import cv2
    wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (1280, 720))
    base = [picture(720, 1280, 100 + k, sigma) for k in range(16)]
    for i in range(n):
        wr.write(np.roll(base[i % 16], 7 * i, axis=1))
    wr.release()


def device_decode(path, sessions, batch=32):
    t = time.perf_counter()
    pending, n = [], 0
    for i, (packets, first, nv) in enumerate(extract.FrameBatches(path, batch=batch, depth=5, pad_last=True,
                                                                  decode="device")):
        if len(pending) == len(sessions):
            pending.pop(0).status()                # that session's decode has finished: it takes the next batch
        pending.append(jpeg.DeviceFrames(sessions[i % len(sessions)], packets, first))
        n += nv
    for d in pending:
        d.status()
    return n / (time.perf_counter() - t)


def cv2_decode(path, workers, batch=32):
    t = time.perf_counter()
    n = sum(len(fr) for fr, _ in extract.FrameBatches(path, batch=batch, depth=5, workers=workers))
    return n / (time.perf_counter() - t)


def job(fn, path, decode, tmp):
    t = time.perf_counter()
    fn(path, tmp, decode)
    return extract.frame_count(path) / (time.perf_counter() - t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_device_decode.json"))
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs the GPU"
    body = Batch_body(O.make_weights("body", 0))
    hand = Batch_hand(O.make_weights("hand", 5, "kaiming"))
    sessions = [body.net.session(), body.net.session()]
    res = {"card": card(), "frames": a.frames, "clips": {}}
    with tempfile.TemporaryDirectory() as d:
        def body_job(path, tmp, dec):
            kw = {"decode": "device"} if dec == "device" else {"decode_workers": 4}
            extract.batch_body_extraction(path, os.path.join(d, "b.pkl"), 32, None, body, log=lambda m: None, **kw)

        def bodyhand_job(path, tmp, dec):
            kw = {"decode": "device"} if dec == "device" else {"decode_workers": 4}
            extract.batch_bodyhand_extraction(path, os.path.join(d, "b.pkl"), os.path.join(d, "h.pkl"), 32, None, body,
                                              hand, log=lambda m: None, **kw)
        for name, sigma in (("high_detail_sigma2", 2.0), ("low_detail_sigma8", 8.0)):
            path = os.path.join(d, name + ".avi")
            write_clip(path, a.frames, sigma)
            sizes = packet_sizes(path)
            r = {"packet_bytes_mean": float(np.mean(sizes)), "packet_bytes_max": int(max(sizes))}
            device_decode(path, sessions)                              # warm-up
            body_job(path, d, "device")
            bodyhand_job(path, d, "device")
            body_job(path, d, "cv2")
            for key in ("decode_device_fps", "decode_cv2_1thread_fps", "decode_cv2_4threads_fps", "batch_body_device_fps",
                        "batch_body_cv2x4_fps", "batch_bodyhand_device_fps", "batch_bodyhand_cv2x4_fps"):
                r[key] = []
            for _ in range(2):
                r["decode_device_fps"].append(device_decode(path, sessions))
                r["decode_cv2_1thread_fps"].append(cv2_decode(path, 1))
                r["decode_cv2_4threads_fps"].append(cv2_decode(path, 4))
                r["batch_body_device_fps"].append(job(body_job, path, "device", d))
                r["batch_body_cv2x4_fps"].append(job(body_job, path, "cv2", d))
                r["batch_bodyhand_device_fps"].append(job(bodyhand_job, path, "device", d))
                r["batch_bodyhand_cv2x4_fps"].append(job(bodyhand_job, path, "cv2", d))
            # kernel shares of the device decode, in a profiled run of its own
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                device_decode(path, sessions)
            k = {}
            for e in prof.key_averages():
                m = re.search(r"jpeg_\w+_kernel", e.key)
                if m:
                    k[m.group(0)] = k.get(m.group(0), 0) + getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0))
            total = sum(k.values())
            r["kernel_us"] = k
            r["entropy_share"] = (sum(v for n, v in k.items() if "entropy" in n) / total) if total else None
            res["clips"][name] = r
            print(name, json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
