"""Builds pytorch_openpose_b200/libopenpose_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m pytorch_openpose_b200.build [--force]

No torch headers are involved: the library exposes the plain C ABI of include/openpose_b200.h and is loaded
with ctypes (pytorch_openpose_b200/_lib.py)."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libopenpose_b200.so")
BUILD = os.path.join(HERE, "build")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"]
# units whose float64 arithmetic must round exactly like numpy/scipy: no FMA contraction
EXACT = {"peaks.cu", "paf.cu", "hand.cu", "prepost.cu", "pose.cu", "track.cu"}
SOURCES = ["conv_tc.cu", "conv_patch.cu", "conv_pair.cu", "conv_tail.cu", "conv_simt.cu", "prepost.cu", "peaks.cu", "paf.cu", "hand.cu", "pose.cu", "track.cu", "net.cu", "api.cu"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = _nvcc()
    os.makedirs(BUILD, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "openpose_b200.h"))
    headers.append(os.path.abspath(__file__))
    jobs = []
    objs = []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        obj = os.path.join(BUILD, src.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [path] + headers):
            cmd = [nvcc] + ARCH + COMMON + (["--fmad=false"] if src in EXACT else []) + ["-c", path, "-o", obj]
            jobs.append(cmd)

    def run(cmd):
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), r.stderr))
        return r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for err in ex.map(run, jobs):
                if verbose and err.strip():
                    print(err)
    if jobs or force or _stale(OUT, objs):
        run([nvcc] + ARCH + ["-shared", "-o", OUT] + objs + ["-Xcompiler", "-fPIC", "-cudart", "static"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
