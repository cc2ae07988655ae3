"""Build libpyrope_gpu.so in-tree with nvcc for sm_100a (B200).  No GPU is needed to compile."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libpyrope_gpu.so")
SOURCES = ["api.cu", "flat.cu", "ivf.cu", "pq.cu", "pq_lm.cu", "ivf_lm.cu", "build.cu", "flat_tc.cu", "coarse_tc.cu", "batcher.cu", "vindex.cu", "formats.cu", "sq8.cu", "sharded.cu", "peer.cu", "extend.cu"]
HEADERS = ["common.cuh", "internal.h", "kernels.h", "exact_arith.cuh", "dotnet_random.h", "../../include/pyrope_gpu.h"]

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
EXTRA = os.environ.get("PYROPE_NVCC_EXTRA", "").split()  # extra nvcc flags for experiments (e.g. a -D switch)
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++",
]


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace(".cu", ".o"))
        if force or _stale(obj, [src] + hdrs + [os.path.abspath(__file__)]):
            cmd = [NVCC] + FLAGS + EXTRA + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0 or verbose:
            sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for " + cmd[-3])

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        list(ex.map(run, jobs))
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in srcs]
    if force or jobs or _stale(LIB, objs):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "/usr/bin/g++"]
        run(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
