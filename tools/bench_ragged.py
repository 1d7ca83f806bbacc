"""Hand() on square crops whose sides differ from crop to crop (util.handDetect's boxes follow the arm), at the default 4
scales.  Prints one JSON line with crops/s for
  - the per-crop loop Hand()(crop): its first pass over sides it has never seen (each new side builds a frame plan of
    tap tables: the per-size cost the loop pays) and a second pass over the same crops;
  - Hand()(list) in ragged batches of 8, 16 and 32 crops (two sessions in flight, as Hand.__call__ chunks);
  - the ceiling: the same number of crops all of the largest side as one equal-size array, in batches of 32.
Workload: 512 seeded crops of blurred noise, sides drawn uniformly from 64..400, pageable host arrays.  Every
configuration is warmed up first (the loop's second pass reuses the first pass's plans); the runs are alternated and
each figure is taken twice.  The ragged rows are checked to equal the loop's rows bit for bit.

    python tools/bench_ragged.py [out.json]"""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2                                                               # noqa: E402
from oracle import openpose_oracle as O                                 # noqa: E402
from pytorch_openpose_b200 import Hand                                  # noqa: E402

N, SIDE_LO, SIDE_HI = 512, 64, 400


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


rng = np.random.default_rng(0)
sides = [int(v) for v in rng.integers(SIDE_LO, SIDE_HI + 1, N)]
crops = [cv2.GaussianBlur(rng.integers(0, 256, (w, w, 3), dtype=np.uint8), (0, 0), 2) for w in sides]
ceiling = np.stack([cv2.resize(c, (max(sides), max(sides))) for c in crops])
weights = O.make_weights("hand", 5, "kaiming")


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return N / (time.perf_counter() - t0), out


loop_hand = Hand(weights)
first_rate, loop_rows = timed(lambda: np.stack([loop_hand(c) for c in crops]))       # sides never seen before
hands = {}
for b in (8, 16, 32):
    hands[b] = Hand(weights)
    hands[b].MAX_BATCH = b
    assert np.array_equal(hands[b](crops), loop_rows), b                               # warm-up and parity
ceil_hand = Hand(weights)
ceil_hand(ceiling)

runs = {"loop": lambda: np.stack([loop_hand(c) for c in crops]), "ceiling_equal_size_32": lambda: ceil_hand(ceiling)}
for b in (8, 16, 32):
    runs["ragged_%d" % b] = (lambda h: lambda: h(crops))(hands[b])
rates = {k: [] for k in runs}
for rep in range(2):
    for k, fn in runs.items():
        r, out = timed(fn)
        if k != "ceiling_equal_size_32":
            assert np.array_equal(out, loop_rows), k
        rates[k].append(round(r, 1))

out = dict(gpu_info())
out.update({"crops": N, "sides": [SIDE_LO, SIDE_HI], "distinct_sides": len(set(sides)), "scales": loop_hand.scale_search,
            "loop_first_pass_crops_per_s": round(first_rate, 1),
            "loop_first_pass_ms_per_crop": round(1e3 / first_rate, 3)})
out.update({k + "_crops_per_s": v for k, v in rates.items()})
line = json.dumps(out)
print(line)
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        f.write(line + "\n")
