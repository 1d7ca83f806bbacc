"""Cost of the exact component choice of the hand post-processing (csrc/hand.cu, hand_select_kernel) on one B200.

One 736 x 736 crop whose first two key-point maps hold 200 identical blobs (values 1e-12 ... 1): every component ties,
so every one of them takes the exact path.  The same call on the same maps with the blobs scaled apart (no contenders)
is the fast path.  Both run through opb_hand_debug_post (six launches, host synchronise at the end); CUDA events around
each call, medians over repeated calls, alternating the two.  The difference is the exact path's time."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from tests.test_gpu_hand_post import many_copies, post   # noqa: E402


def main(reps=20):
    tied = many_copies()
    apart = tied.copy()
    for p in (0, 1):
        ys, xs = np.nonzero(apart[0, p])
        apart[0, p, ys, xs] *= (1.0 + 1e-3 * ((ys // 46) * 15 + xs // 46)).astype(np.float32)   # one scale per blob
    res = {}
    for name, m in (("tied_200", tied), ("apart_200", apart)):
        post(m)                                        # warm-up
    times = {"tied_200": [], "apart_200": []}
    for _ in range(reps):
        for name, m in (("tied_200", tied), ("apart_200", apart)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            post(m)
            b.record()
            torch.cuda.synchronize()
            times[name].append(a.elapsed_time(b))
    for k, v in times.items():
        res[k + "_ms"] = float(np.median(v))
    res["exact_path_ms"] = res["tied_200_ms"] - res["apart_200_ms"]
    q = "--query-gpu=name,power.limit"
    res["gpu"] = subprocess.run(["nvidia-smi", q, "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(json.dumps({"metric": "hand_exact_path", "results": res}))


if __name__ == "__main__":
    main()
