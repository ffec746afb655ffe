"""Build libbmm_b200.so in-tree with nvcc for sm_100a (no torch, no JIT cache).

    python -m bmm_mcmc_b200.build [--force]
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libbmm_b200.so")
SOURCES = ["capi.cu", "dist.cu", "kern_full.cu", "kern_collapsed.cu", "kern_stephens.cu", "kern_finalize.cu",
           "kern_big.cu", "kern_big_ws.cu", "kern_big_lp.cu", "kern_big_counts.cu", "kern_big_relabel.cu", "kern_big_cost_tc.cu", "kern_big_ws_relabel.cu", "kern_predict.cu", "kern_waic_tc.cu", "kern_loo.cu",
           "host_widen.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
              "--expt-extended-lambda"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    return "nvcc"


def _deps():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(HERE, "..", "include", "bmm_capi.h"))
    return max(os.path.getmtime(h) for h in hdrs)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    hdr_m = _deps()
    jobs = []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, os.path.splitext(s)[0] + ".o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_m):
            jobs.append((src, obj))
    nvcc = _nvcc()

    def cc(job):
        src, obj = job
        if src.endswith(".cpp"):
            cmd = ["g++", "-O3", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-mavx2", "-pthread", "-c", src, "-o", obj]
        else:
            cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stderr))
        if verbose and r.stderr:
            sys.stderr.write(r.stderr)

    if jobs:
        with ThreadPoolExecutor(max_workers=8) as ex:
            list(ex.map(cc, jobs))
    objs = [os.path.join(OBJ, os.path.splitext(s)[0] + ".o") for s in srcs]
    if jobs or not os.path.exists(LIB):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl", "-lpthread"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
