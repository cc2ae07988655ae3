"""What a Build costs at the C5-like shape of tests/test_gpu_fullshape.py, and how often the shortlist gate of coarse
assignment sends a row to the exhaustive redo there.

Each measurement runs in a child process: 2 M uniform rows (fill_uniform_device, seed 42), IVF_PQ, dim 128, m 16,
k 256, nlist 16,384, training bounded to 4 x nlist rows and 2 Lloyd iterations (as test_gpu_fullshape), then
pyrope_index_build timed with the host clock (it returns after its device work; a synchronise follows).  With several
--lib paths (builds of the library to compare) the children alternate, --repeats rounds, and each prints a hash of the
centroids, codebooks and lists so that equal outputs can be checked.  --redo-sample N emulates the gate
(tests/test_gpu_build_regimes.py: 3xTF32 proxy, rounding-bound gate and the relative margin it replaced) on the first N
rows against the trained centroids; that fraction is an emulation, not a device count.  Prints one JSON line with the
card's name and power limit.

    python profiles/build_c5_shape.py [--lib A.so --lib B.so] [--repeats 3] [--redo-sample 4096] [--out F]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DIM, N, NLIST, M = 128, 2_000_000, 16384, 16


def child(lib, redo_sample):
    import numpy as np
    import torch

    from pyrope_b200 import _lib
    if lib:
        _lib.LIB_PATH = os.path.abspath(lib)
    import pyrope_b200 as pg
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this script measures on the device and has no CPU fallback")
    _lib.check(pg.load().pyrope_gpu_init(0))
    ix = pg.GpuIndex(pg.IVF_PQ, DIM, pg.L2, nlist=NLIST, m=M, k=256)
    ix.set_train_params(4 * NLIST, 2)
    ix.reserve(N)
    stage = torch.empty(N * DIM, dtype=torch.float32, device="cuda")
    _lib.fill_uniform_device(stage.data_ptr(), N * DIM, 42, 0, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ix.add_device(stage.data_ptr(), N)
    head = stage[:max(redo_sample, 1) * DIM].view(-1, DIM).cpu().numpy()
    del stage
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ix.build()
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    cent = ix.centroids()
    cb, ks = ix.codebooks()
    off, rows, codes = ix.lists()
    h = hashlib.sha256()
    for a in (cent, cb, ks, off, rows, codes):
        h.update(np.ascontiguousarray(a).tobytes())
    out = {"build_s": round(build_s, 3), "outputs_sha256": h.hexdigest()[:16]}
    if redo_sample:
        from oracle import pyoracle as orc
        from tests.test_gpu_build_regimes import KPRIME, new_gate, old_gate, proxy_scores
        P, A = proxy_scores(head, cent, orc.L2)
        redo = {"new": 0, "old": 0}
        for i in range(len(head)):
            order = np.argsort(-P[i], kind="stable")[:KPRIME]
            p0, plast = P[i, order[0]], P[i, order].min()
            redo["new"] += not new_gate(p0, plast, head[i], A, orc.L2)
            redo["old"] += not old_gate(p0, plast, head[i], A, orc.L2)
        out["emulated_redo_fraction"] = {k: v / len(head) for k, v in redo.items()}
        out["redo_sample_rows"] = len(head)
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=None, help="library to load (repeatable); default: the tree's")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--redo-sample", type=int, default=0)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child is not None:
        return child(args.child, args.redo_sample)

    from profiles.sharded_delta_step import gpu_info
    libs = args.lib or [""]
    runs = {lib or "tree": [] for lib in libs}
    for r in range(args.repeats):
        for lib in libs:
            cmd = [sys.executable, os.path.abspath(__file__), "--child", lib,
                   "--redo-sample", str(args.redo_sample if r == 0 else 0)]
            res = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
            if res.returncode != 0:
                raise SystemExit(f"child {lib or 'tree'} failed:\n{res.stdout}\n{res.stderr}")
            runs[lib or "tree"].append(json.loads(res.stdout.strip().splitlines()[-1]))
    summary = {}
    for name, rs in runs.items():
        summary[name] = {"build_s_median": statistics.median(x["build_s"] for x in rs),
                         "build_s": [x["build_s"] for x in rs],
                         "outputs_sha256": sorted({x["outputs_sha256"] for x in rs})}
        for x in rs:
            if "emulated_redo_fraction" in x:
                summary[name]["emulated_redo_fraction"] = x["emulated_redo_fraction"]
                summary[name]["redo_sample_rows"] = x["redo_sample_rows"]
    line = json.dumps({"shape": {"rows": N, "dim": DIM, "nlist": NLIST, "m": M, "train_rows": 4 * NLIST, "iters": 2},
                       **gpu_info(), "runs": summary})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
