#!/usr/bin/env python
"""Benchmark of the OpenPose hot path (BASELINE.json: body-pose frames/s at 720p, 4 scales).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--frames-per-step F]
                    [--dump-outputs DIR]

A step is one pass of the whole Body path (preprocess at 4 scales -> CNN -> upsample/average -> Gaussian+NMS ->
PAF scoring / matching / assembly) over F synthetic 1280x720 frames on every rank, submitted as F/B batches of B
frames (one launch per CNN layer per batch) round-robin over a few streams; frames are independent, so ranks never
exchange data (weak scaling, no collective on the data path).  Rank 0 prints ONE
JSON line.  `value` is measured with the frames already resident in HBM; `e2e` goes through the same public
`Body` API with pinned HOST frames, the host->device copy of every frame and the device->host read of every
result inside the timed region.  `--impl reference` times the CPU restatement of the reference (oracle/) on the
host cores instead.  `--dump-outputs DIR` writes the results of the last timed step (see dump_outputs); inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 720, 1280
SCALES = (0.5, 1.0, 1.5, 2.0)
METRIC = "body_pose_frames_per_sec_720p_4scale"
GFLOP_PER_FRAME = 3634.8          # SURVEY.md 8d: algorithmic conv FLOPs of the body net at the four padded sizes
POOL_FRAMES = 80                  # 80 x 2.76 MB = 221 MB of distinct inputs (> 126 MB L2)
REF_POOL_FRAMES = 12              # distinct frames of the host-side reference leg, reused modulo the pool
DUMP_LIMIT = 64 << 20             # bytes --dump-outputs may write


def rank_info():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def synth_frames(n, seed):
    """Structured synthetic frames (blurred noise): cheap to make, not constant."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (n, H // 8, W // 8, 3), dtype=np.uint8)
    return np.ascontiguousarray(np.repeat(np.repeat(base, 8, 1), 8, 2))


def dump_outputs(d, results):
    """Writes one step's per-frame (candidate, subset) results, what Body hands its caller, as float64 .npy files:
    candidate.npy (N, 4) and subset.npy (M, 20) hold the rows of all written frames in frame order, and
    candidate_rows.npy / subset_rows.npy how many rows belong to each of them.  frame_index.npy names the frames of
    the step that were written: all of them, or a fixed seeded sample when the whole step exceeds DUMP_LIMIT.
    An array without rows is not written: its row counts, all zero, already say everything it holds (random-init
    weights find candidates but assemble no person, so subset.npy is usually absent)."""
    cands = [np.asarray(c, dtype=np.float64).reshape(-1, 4) for c, _ in results]
    subs = [np.asarray(s, dtype=np.float64).reshape(-1, 20) for _, s in results]
    n = len(results)
    keep = np.arange(n)
    nbytes = np.array([c.nbytes + s.nbytes + 3 * 8 for c, s in zip(cands, subs)])
    if nbytes.sum() > DUMP_LIMIT:
        perm = np.random.default_rng(0).permutation(n)
        keep = np.sort(perm[:np.searchsorted(np.cumsum(nbytes[perm]), DUMP_LIMIT, side="right")])
    os.makedirs(d, exist_ok=True)
    arrays = {"candidate": np.concatenate([cands[i] for i in keep] or [np.empty((0, 4))]),
              "subset": np.concatenate([subs[i] for i in keep] or [np.empty((0, 20))]),
              "candidate_rows": np.array([len(cands[i]) for i in keep], dtype=np.float64),
              "subset_rows": np.array([len(subs[i]) for i in keep], dtype=np.float64),
              "frame_index": keep.astype(np.float64)}
    for name, a in arrays.items():
        if a.size:
            np.save(os.path.join(d, name + ".npy"), a)


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nme, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p["bf16_tflops_sustained"], p["hbm_gbs"], "measured (MEASURED_PEAKS.json, sustained bf16)"
    except Exception:
        return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def cpu_reference_frames(n_frames, threads):
    """The reference's algorithm on the host cores: the oracle's Body.__call__ restatement, torch CPU fp32 convs,
    cv2 resizes, scipy-exact Gaussian, Python PAF loops vectorised per limb.  Returns the list of seconds per frame
    and the (candidate, subset) of the last frame."""
    import torch
    from oracle import openpose_oracle as O
    torch.set_num_threads(threads)
    sd = O.make_weights("body", 0)
    frames = synth_frames(max(1, min(n_frames, REF_POOL_FRAMES)), 123)
    times, out = [], None
    for i in range(n_frames):
        t0 = time.perf_counter()
        out = O.body_call(frames[i % len(frames)], sd, SCALES, use_cv2=True)
        times.append(time.perf_counter() - t0)
    return times, out


def run_reference(args):
    rank, _, world = rank_info()
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    warm = min(args.warmup, 1)                   # one 720p 4-scale frame is ~10 s of CPU work
    steps = args.steps
    times, last = cpu_reference_frames(warm + steps, threads)
    sec = float(np.sum(times[warm:]))
    fps = steps / sec
    line = {"metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": 1e3 * sec / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "Body() 4-scale [0.5,1.0,1.5,2.0] on synthetic 1280x720 frames, random-init bodypose_model",
                       "frames_per_step": 1, "note": "warmup capped at 1: one frame is ~10 s on the host"},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                             "sample": "%d full frames (oracle restatement of src/body.py; the reference checkout is not on the GPU box)" % steps},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [last])
    print(json.dumps(line), flush=True)



# ---- further BASELINE.json configurations, measured through the public API at every N (all ranks run, max over ranks) ----
def extra_hand_c3(local, barrier, max_over_ranks, world):
    """config 3: Hand() on 256 synthetic 368x368 crops (host memory in, key points out), 4 scales like src/hand.py:26
    and one scale."""
    import torch
    from pytorch_openpose_b200 import Hand
    from pytorch_openpose_b200.model import random_checkpoint
    crops = np.random.default_rng(7).integers(0, 256, (256, 368, 368, 3), dtype=np.uint8)
    sd = random_checkpoint("hand", 0)
    out = {"workload": "Hand()(crops): 256 synthetic 368x368 crops from host memory, wall clock incl. H2D / D2H"}
    for tag, scales, gflop in (("4scale", [0.5, 1.0, 1.5, 2.0], 1547.82), ("1scale", [1.0], 206.38)):
        hand = Hand(sd, scale_search=scales, device=local)
        hand(crops)                                     # builds the plans
        reps = 2 if tag == "4scale" else 4
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            hand(crops)
        torch.cuda.synchronize()
        dt = max_over_ranks((time.perf_counter() - t0) / reps)
        out[tag] = {"crops_per_s": round(256 * world / dt, 1), "ms_per_256": round(dt * 1e3, 2),
                    "conv_tflops_per_gpu": round(gflop * 256 / dt * 1e-3, 1)}
        del hand
    peak, _, _ = measured_peaks()
    out["roofline"] = {"bound": "tensor", "achieved": out["4scale"]["conv_tflops_per_gpu"], "peak": peak, "unit": "TFLOP/s",
                       "frac": round(out["4scale"]["conv_tflops_per_gpu"] / peak, 3),
                       "note": "whole call incl. copies and post-processing over the algorithmic conv FLOPs (1547.8 GFLOP/crop)"}
    return out


def extra_bodyhand_c4(local, rank, barrier, max_over_ranks, world, streams=2, B=8, F=32, steps=4):
    streams = int(os.environ.get("OPB_C4_STREAMS", streams))
    """config 4: 720p stream, body (4 scales) + two hands (4 scales) per frame through motion.PoseEstimator: the hand
    crops are cut (the left one mirrored) from the frame already on the device, all 2 * B crops of a batch run as one
    ragged hand batch, PoseMat (60, 3) per frame is the only result read back.  Random-init weights find no person, so
    the two hand boxes are fixed 184x184 boxes (SURVEY.md 8d C4) instead of handDetect's."""
    import torch
    from pytorch_openpose_b200 import Body, Hand, motion
    from pytorch_openpose_b200.model import random_checkpoint
    body = Body(random_checkpoint("body", 0), scale_search=SCALES, device=local)
    hand = Hand(random_checkpoint("hand", 0), device=local)
    est = motion.PoseEstimator(body, hand)
    pairs = est.sessions(streams)
    pool = torch.from_numpy(synth_frames(32, 77 + rank)).pin_memory()
    frames = pool.numpy()
    boxes = np.tile(np.array([[400, 300, 184], [700, 300, 184]], dtype=np.int32), (B, 1, 1))

    def step(i):
        inflight = [False] * streams
        for b in range(F // B):
            si = b % streams
            if inflight[si]:
                est.collect(pairs[si])
            idx = (i * F + b * B) % 32
            est.submit_batch(frames[idx:idx + B], pairs[si], where=2, fixed_boxes=boxes)
            inflight[si] = True
        out = None
        for si in range(streams):
            if inflight[si]:
                out = est.collect(pairs[si])
        return out

    for i in range(2):
        step(i)
    barrier()
    pairs[0][0].mark(0)
    for i in range(steps):
        out = step(2 + i)
    for bs, _ in pairs:
        bs.mark(1)
    torch.cuda.synchronize()
    ms = max_over_ranks(max(pairs[0][0].elapsed_ms(0, bs, 1) for bs, _ in pairs))
    n = F * steps * world
    peak, _, _ = measured_peaks()
    tf = 6730.4 * F * steps / ms
    return {"value": round(n / (ms * 1e-3), 1), "unit": "frames/s", "ms_per_frame_per_gpu": round(ms / (F * steps), 3),
            "conv_tflops_per_gpu": round(tf, 1),
            "roofline": {"bound": "tensor", "achieved": round(tf, 1), "peak": peak, "unit": "TFLOP/s", "frac": round(tf / peak, 3)},
            "h2d_bytes_per_frame": H * W * 3, "d2h_bytes_per_frame": 60 * 3 * 8 + 86144,
            "hand_key_points_found": int((out[:, 18:, 2] > 0).sum()),
            "workload": "body 4-scale + two 184x184 hand boxes 4-scale per 720p frame, pinned host frames in, PoseMat out; "
                        "crops, mirroring, resize and the ragged hand batch on the device (CUDA events over %d frames per GPU)"
                        % (F * steps)}


def extra_e2e_decode(local, rank, barrier, max_over_ranks, world, n_frames=256):
    """Decode-inclusive leg: MJPG 720p file -> cv2.VideoCapture threads -> pinned batch ring -> Body 4-scale -> pose
    track (pytorch_openpose_b200.extract, the reference's Extract_MotionData_from_Video).  Every rank decodes its own
    file at the same time with cpu_count / world decoder threads (at most 4), so the figure shows whether host decode
    bends the 1 -> 8 curve.  Wall clock, max over ranks."""
    import tempfile
    import cv2
    import torch
    from pytorch_openpose_b200 import Body, extract
    from pytorch_openpose_b200.model import random_checkpoint
    d = tempfile.mkdtemp(prefix="opb_bench_%d_" % rank)
    path = os.path.join(d, "v.avi")
    wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (W, H))
    base = synth_frames(8, 500 + rank)
    for i in range(n_frames):
        wr.write(np.roll(base[i % 8], 7 * i, axis=1))
    wr.release()
    workers = max(1, min(4, (os.cpu_count() or 1) // world))
    body = Body(random_checkpoint("body", 0), scale_search=SCALES, device=local)
    quiet = lambda m: None
    extract.extract_motion_from_video(path, os.path.join(d, "w.pkl"), None, body, mode="body", batch=8, sessions=3,
                                      log=quiet, decode_workers=workers)                  # plans + pinned rings
    passes = []
    for rep in range(3):                # 256 frames take ~0.8 s of wall clock: one hiccup of the host is 20 % -> median of 3 passes
        barrier()
        t0 = time.perf_counter()
        mat = extract.extract_motion_from_video(path, os.path.join(d, "o%d.pkl" % rep), None, body, mode="body", batch=8,
                                                sessions=3, log=quiet, decode_workers=workers)
        torch.cuda.synchronize()
        passes.append(max_over_ranks(time.perf_counter() - t0))
    dt = sorted(passes)[1]
    # decode alone, same threads, all ranks at once
    barrier()
    t0 = time.perf_counter()
    n = sum(len(item[0]) for item in extract.FrameBatches(path, None, batch=8, depth=5, pinned=True, workers=workers))
    ddt = max_over_ranks(time.perf_counter() - t0)
    import shutil
    shutil.rmtree(d, ignore_errors=True)
    return {"value": round(len(mat) * world / dt, 1), "unit": "frames/s", "decode_only_frames_per_s": round(n * world / ddt, 1),
            "decoder_threads_per_rank": workers, "host_cores": os.cpu_count(), "frames_per_rank": int(len(mat)),
            "passes_frames_per_s": [round(len(mat) * world / t, 1) for t in passes],
            "workload": "720p MJPG file per rank -> decode threads -> pinned ring -> Body 4-scale -> pose track file; "
                        "wall clock, median of 3 passes"}


def run_ours(args):
    import torch
    from pytorch_openpose_b200 import Body, _lib
    from pytorch_openpose_b200.model import random_checkpoint      # random-init weights, seed 0 (no checkpoints offline)
    rank, local, world = rank_info()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner to STDOUT at NCCL_DEBUG=VERSION and WARN, which some images export: the contract
        # is one JSON line on stdout, so NCCL logging is off unless the caller asks (OPB_NCCL_DEBUG=INFO shows NVLS etc.)
        if "OPB_NCCL_DEBUG" in os.environ:
            os.environ["NCCL_DEBUG"] = os.environ["OPB_NCCL_DEBUG"]
        else:
            os.environ.pop("NCCL_DEBUG", None)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    F, K, Wm = args.frames_per_step, args.steps, args.warmup
    body = Body(random_checkpoint("body", 0), scale_search=SCALES, device=local)
    sessions = [body.net.session() for _ in range(args.streams)]
    frames_host = torch.from_numpy(synth_frames(POOL_FRAMES, 1000 + rank)).pin_memory()
    frames_dev = frames_host.cuda()
    host_np = frames_host.numpy()
    torch.cuda.synchronize()

    B = args.batch
    assert F % B == 0 and POOL_FRAMES % B == 0, "frames-per-step and the frame pool must be multiples of --batch"

    def step(step_idx, device_resident):
        """F frames as F/B batches of B consecutive pool frames, round-robin over the sessions (streams).
        Returns the (candidate, subset) of every frame, in frame order."""
        pending = [None] * len(sessions)             # batch in flight on each session
        results = [None] * (F // B)
        for b in range(F // B):
            si = b % len(sessions)
            if pending[si] is not None:
                results[pending[si]] = body.collect_batch(sessions[si])
            idx = (step_idx * F + b * B) % POOL_FRAMES
            if device_resident:
                body.submit_batch((frames_dev[idx].data_ptr(), (B, H, W)), sessions[si], where=1)
            else:
                body.submit_batch(host_np[idx:idx + B], sessions[si], where=2)
            pending[si] = b
        for si, b in enumerate(pending):
            if b is not None:
                results[b] = body.collect_batch(sessions[si])
        return [r for batch in results for r in batch]

    def timed(device_resident):
        for w in range(Wm):
            step(w, device_resident)
        barrier()
        l0 = _lib.launch_count(local)
        sessions[0].mark(0)
        for k in range(K):
            out = step(Wm + k, device_resident)
        for s in sessions:
            s.mark(1)
        torch.cuda.synchronize()
        ms = max(sessions[0].elapsed_ms(0, s, 1) for s in sessions)
        launches = _lib.launch_count(local) - l0
        barrier()
        return max_over_ranks(ms), launches, out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev, launches, last = timed(True)
    clocks = sampler.stop() if rank == 0 else None
    ms_e2e, _, _ = timed(False)

    # ---- roofline of the dominant kernel (tcgen05 implicit-GEMM conv), serialised profiled frames ----
    roof = None
    stages = {}
    if rank == 0:
        s0 = sessions[0]
        s0.set_profiling(True)
        tc_ms, tc_gf, tc_n, n_prof = 0.0, 0.0, 0, 4
        for i in range(n_prof):
            idx = (i * B) % POOL_FRAMES
            body.submit_batch((frames_dev[idx].data_ptr(), (B, H, W)), s0, where=1)    # the benchmarked batch shape
            body.collect_batch(s0)
            for name, ms, gf in s0.profile():
                key = name.split(":")[0]
                stages[key] = stages.get(key, 0.0) + ms / (n_prof * B)
                if key == "conv_tc128":
                    tc_ms += ms
                    tc_gf += gf
                    tc_n += 1
        if args.layers:
            per = {}
            for name, ms, gf in s0.profile():
                a = per.setdefault(name, [0.0, 0.0])
                a[0] += ms
                a[1] += gf
            with open(args.layers, "w") as f:
                f.write("step,ms,gflop,tflops\n")
                for name, (ms, gf) in per.items():
                    f.write("%s,%.4f,%.2f,%.1f\n" % (name, ms, gf, gf / ms if ms > 0 else 0.0))
        s0.set_profiling(False)
        peak, hbm, how = measured_peaks()
        achieved = tc_gf / tc_ms if tc_ms > 0 else 0.0            # GFLOP/ms == TFLOP/s
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        except Exception:
            pass
        roof = {"bound": "tensor",
                "kernel": "tcgen05 implicit-GEMM conv, N=128 variants (conv_pair_kernel<128> cta_group::2 for 3x3/7x7 incl. conv1_2 in its wide-pixel form, conv_tc_kernel<128> for 1x1): "
                          "mean over its %d launches per batch of %d frames" % (tc_n // n_prof, B),
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "peak_source": how,
                "traffic": traffic, "traffic_note": "DRAM bytes of the ncu-captured 7x7 stage launch (profiles/roofline_traffic.json)",
                "gflop_per_launch": tc_gf / max(tc_n, 1), "ms_per_launch": tc_ms / max(tc_n, 1),
                "gflop_per_frame": tc_gf / (n_prof * B), "ms_per_frame": tc_ms / (n_prof * B),
                "measured_over": "%d serialised profiled batches of %d frames after the timed region (CUDA events around every launch)" % (n_prof, B),
                "note": "peak is the driver's cuBLAS bf16 measurement (sustained, power-capped) for this pool; boxes differ by "
                        "a few percent, so frac can land slightly above 1"}

    # ---- BASELINE.json's second metric: PAF-grouping ms/frame on the crowded synthetic scene (50 people) ----
    grouping = None
    if rank == 0 and not args.no_grouping:
        import ctypes
        from oracle import openpose_oracle as O        # checker / CPU leg only: the synthetic 50-person scene and its CPU timing
        heat50, paf50, _ = O.synthetic_scene(H, W, (10, 5), seed=0)
        d_heat = torch.from_numpy(np.ascontiguousarray(heat50.transpose(2, 0, 1), dtype=np.float32)).cuda()
        d_paf = torch.from_numpy(np.ascontiguousarray(paf50.transpose(2, 0, 1), dtype=np.float32)).cuda()
        torch.cuda.synchronize()
        ms, nc, ns = ctypes.c_float(), ctypes.c_int(), ctypes.c_int()
        _lib.check(_lib.lib().opb_bench_grouping(_lib.context(local), d_heat.data_ptr(), d_paf.data_ptr(), H, W, 50,
                                                 ctypes.byref(ms), ctypes.byref(nc), ctypes.byref(ns)))
        grouping = {"value": ms.value, "unit": "ms/frame", "candidates": nc.value, "persons": ns.value,
                    "workload": "synthetic 1280x720 maps, 50 people, 47.5 k limb pairs: Gaussian + NMS + PAF scoring + matching + assembly"}
        if world == 1 and not args.no_cpu_baseline:
            t0 = time.perf_counter()
            O.body_postprocess(heat50, paf50, H)
            grouping["cpu_port_ms"] = 1e3 * (time.perf_counter() - t0)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:        # reported at N=1 only
        threads = os.cpu_count() or 1
        t, _ = cpu_reference_frames(2, threads)
        cpu = {"value": 2.0 / float(np.sum(t)), "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": "2 full 720p 4-scale frames through the oracle restatement of src/body.py (no warm-up)"}

    extras = {}
    n_streams = len(sessions)
    if not args.no_extras:
        n_streams = len(sessions)
        del sessions, frames_dev
        torch.cuda.empty_cache()
        for name, fn in (("hand_c3", lambda: extra_hand_c3(local, barrier, max_over_ranks, world)),
                         ("bodyhand_c4", lambda: extra_bodyhand_c4(local, rank, barrier, max_over_ranks, world)),
                         ("e2e_decode", lambda: extra_e2e_decode(local, rank, barrier, max_over_ranks, world))):
            try:
                extras[name] = fn()
            except Exception as e:                      # an extra leg must never cost the headline line
                extras[name] = {"error": "%s: %s" % (type(e).__name__, e)}
            barrier()

    if rank == 0:
        total_frames = F * K * world
        d2h = F * (32 * 4 + 2048 * 4 * 8 + 128 * 20 * 8)    # per frame: one FrameResults block (counts + first candidate / subset rows)
        line = {"metric": METRIC, "value": total_frames / (ms_dev * 1e-3), "unit": "frames/s", "n_gpus": world,
                "steps": K, "warmup": Wm, "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "Body() 4-scale [0.5,1.0,1.5,2.0] on synthetic 1280x720 frames, random-init bodypose_model",
                           "frames_per_step": F, "frames_per_batch": B, "streams": n_streams,
                           "parallelism": "frame-sharded replicas x%d" % world,
                           "l2": "pool of %d distinct frames (221 MB) and ~1 GB of activations per frame exceed the 126 MB L2" % POOL_FRAMES},
                "e2e": {"value": total_frames / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": F * H * W * 3,
                        "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / K},
                "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
                "paf_grouping": grouping, "extra": extras,
                "stage_ms_per_frame": {k: round(v, 4) for k, v in stages.items()}}
        # HBM-bound stages (SURVEY.md 8d): algorithmic bytes per frame / measured stage time vs the measured copy bandwidth
        px_in = sum(hp * wp for hp, wp in ((184, 328), (368, 656), (552, 984), (736, 1312)))
        px_out = sum(a * b for a, b in ((23, 41), (46, 82), (69, 123), (92, 164)))
        alg_mb = {"preprocess": (H * W * 3 + px_in * 3) / 1e6,                        # uint8 frame in, uint8 padded scales out
                  "conv_first": (px_in * 3 + px_in * 64 * 2) / 1e6,                    # conv1_1: K = 27, output-write bound
                  # fused upsample + smoothing + NMS: the low-resolution heat maps (24-channel fp32 pixels) are read once
                  # by the tile-bound pass and once by the peak kernel; nothing full-resolution is written
                  "find_peaks": 2 * px_out * 24 * 4 / 1e6}
        _, hbm_peak, _ = measured_peaks()
        sr = {}
        for name, mb in alg_mb.items():
            if stages.get(name, 0) > 0:
                gbs = mb / stages[name]                                                # MB / ms == GB/s
                sr[name] = {"bound": "hbm", "algorithmic_MB_per_frame": round(mb, 2), "achieved_GBs": round(gbs, 1),
                            "frac_of_hbm_peak": round(gbs / hbm_peak, 3)}
        if "find_peaks" in sr:
            sr["find_peaks"]["bound"] = "issue"
            sr["find_peaks"]["note"] = ("round 1 wrote 210 MB of full-resolution maps per frame and read 66 MB back (upsample_avg 0.17 ms + "
                                        "smooth_nms 0.11 ms); now the maps are evaluated per tile from the net outputs: DRAM traffic "
                                        "= the algorithmic bytes (ncu: profiles/r02_ncu_prepost_c2_b8.csv), time = fp32 FMAs and index "
                                        "arithmetic of the tiles that can hold a peak")
        sr["paf_group"] = {"bound": "latency", "ms_per_frame": stages.get("paf_group"),
                           "note": "PAF values are sampled on demand (10 samples x 2 channels per candidate pair) from the net "
                                   "outputs: the 140 MB of full-resolution PAF planes per frame are never written"}
        line["stage_roofline"] = sr
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames-per-step", type=int, default=32)
    ap.add_argument("--batch", type=int, default=8, help="frames per batched submit (one launch per CNN layer per batch)")
    ap.add_argument("--streams", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-grouping", action="store_true", help="skip the PAF-grouping leg (50-person scene)")
    ap.add_argument("--no-extras", action="store_true", help="skip the config-3 / config-4 / decode-inclusive legs")
    ap.add_argument("--layers", default=None, help="write the per-launch profile of one frame to this CSV")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (float64, at most 64 MB; "
                         "arrays without rows are left out)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
