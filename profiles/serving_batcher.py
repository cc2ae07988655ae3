"""What the micro-batcher buys a server whose sessions each search one query at a time.

T threads (16 / 64 / 256) issue single-query Search calls against a string-id Head+Tail, the object the registry holds:
an IVF_PQ tail (dim 128, m 16, k 256, nlist 4,096, nprobe 64: C5's list parameters over --rows rows instead of 100 M)
under a --head-rows FLAT head.  Three arms, interleaved, each for --calls calls in all:
  (a) direct: every thread calls pyrope_vindex_search with nq = 1 (the shim without a batcher);
  (b) batched: every thread calls VectorIndexBatcher.Search (pyrope_batcher_create_vindex) with topK drawn from
      {1, 5, 10, 20, 50, 100}, so callers of several topK classes share the dispatcher;
  (c) batched, every caller at topK 10: no mix, the most coalescing can reach.
Each arm reports QPS (calls over wall time), p50 / p99 latency per call, and for (b) / (c) the batches and mean batch size.
Every call returns after its result is on the host, so a host clock around the call is its latency.  The host ceiling is
the same threads calling pyrope_version in a loop: Python threads calling through ctypes have a call rate of their own,
and where it is close to an arm's QPS the arm measures Python, not the library.  With several GPUs the batched arms run
again over a tail sharded across all of them.  Prints one JSON line with the card name and power limit.

    python profiles/serving_batcher.py [--rows 2000000] [--head-rows 20000] [--calls 8192] [--rounds 2] [--out F]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from profiles.sharded_delta_step import gpu_info  # noqa: E402

MIX = [1, 5, 10, 20, 50, 100]


def run_threads(T, calls, fn):
    """T threads share `calls` calls of fn(thread, i); returns (wall seconds, per-call latencies in seconds)."""
    per = calls // T
    lat = [[] for _ in range(T)]
    go = threading.Barrier(T + 1)

    def work(t):
        go.wait()
        for i in range(per):
            t0 = time.perf_counter()
            fn(t, i)
            lat[t].append(time.perf_counter() - t0)

    th = [threading.Thread(target=work, args=(t,)) for t in range(T)]
    [x.start() for x in th]
    go.wait()
    t0 = time.perf_counter()
    [x.join() for x in th]
    wall = time.perf_counter() - t0
    return wall, [x for l in lat for x in l]


def summary(wall, lat):
    lat = sorted(lat)
    return {"qps": round(len(lat) / wall, 1), "p50_ms": round(1e3 * lat[len(lat) // 2], 4),
            "p99_ms": round(1e3 * lat[min(len(lat) - 1, int(0.99 * len(lat)))], 4), "calls": len(lat)}


def build_index(vi, rows, head_rows, devices, seed=7):
    params = {"nlist": 4096, "m": 16, "k": 256}
    if devices > 1:
        params["devices"] = devices
    d = vi.create_index("IVF_PQ", 128, vi.VectorMetric.L2, params)
    rng = np.random.default_rng(seed)
    chunk = 100_000
    for lo in range(0, rows, chunk):  # every row enters through the head, as Upserts do, and one Build compacts
        X = rng.random((min(chunk, rows - lo), 128), dtype=np.float32)
        for j in range(X.shape[0]):
            d.Upsert(f"t{lo + j}", X[j])
    d.Build()
    H = rng.random((head_rows, 128), dtype=np.float32)
    for j in range(head_rows):
        d.Upsert(f"h{j}", H[j])
    return d


def measure(vi, d, threads, calls, rounds, direct=True):
    L = vi._lib.load()
    Q = np.random.default_rng(1337).random((4096, 128), dtype=np.float32)
    opts = vi.SearchOptions(NProbe=64)
    out = {}
    for T in threads:
        rng = np.random.default_rng(T)
        ks = rng.choice(MIX, size=calls).astype(int)
        bufs = [(np.zeros(100, np.float32), np.full(100, -1, np.int64), np.zeros(1, np.int32)) for _ in range(T)]

        def arm_direct(t, i):
            s, r, c = bufs[t]
            q = Q[(t * 131 + i) % len(Q)]
            rc = L.pyrope_vindex_search(d._v, 1, q.ctypes.data_as(C.c_void_p), 128, int(ks[(t * 977 + i) % calls]), -1, 64,
                                        s.ctypes.data_as(C.c_void_p), r.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p))
            assert rc == 0, rc
            vi._id_strings(r[:int(c[0])])  # what the shim does with the result, as VectorIndexBatcher does

        def arms_batched(mixed):
            vb = vi.VectorIndexBatcher(d, max_batch=T, max_wait_us=500)

            def fn(t, i):
                vb.Search(Q[(t * 131 + i) % len(Q)], int(ks[(t * 977 + i) % calls]) if mixed else 10, opts)
            return vb, fn

        res = {"direct_topk_mix": [], "batched_topk_mix": [], "batched_topk10": [], "host_ceiling_version": []}
        run_threads(T, min(calls, 4 * T), arm_direct)  # warm-up
        for _ in range(rounds):
            if direct:
                res["direct_topk_mix"].append(summary(*run_threads(T, calls, arm_direct)))
            for name, mixed in (("batched_topk_mix", True), ("batched_topk10", False)):
                vb, fn = arms_batched(mixed)
                run_threads(T, min(calls, 4 * T), fn)  # warm-up of this dispatcher
                b0 = vb.stats()
                s = summary(*run_threads(T, calls, fn))
                b1 = vb.stats()
                nb, nqs = b1["batches"] - b0["batches"], b1["queries"] - b0["queries"]
                s.update({"batches": nb, "mean_batch": round(nqs / max(nb, 1), 2)})
                vb.close()
                res[name].append(s)
            res["host_ceiling_version"].append(summary(*run_threads(T, calls, lambda t, i: L.pyrope_version())))
        best = {k: max(v, key=lambda x: x["qps"]) for k, v in res.items() if v}
        row = {"threads": T, "rounds": res, "best": best,
               "mix_share_of_topk10_qps": round(best["batched_topk_mix"]["qps"] / best["batched_topk10"]["qps"], 3)}
        if direct:
            row["batched_mix_over_direct_qps"] = round(best["batched_topk_mix"]["qps"] / best["direct_topk_mix"]["qps"], 2)
        row["host_ceiling_binds"] = best["batched_topk10"]["qps"] > 0.5 * best["host_ceiling_version"]["qps"]
        out[str(T)] = row
        print(json.dumps({"threads": T, "best": best}), file=sys.stderr, flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=2_000_000)
    ap.add_argument("--head-rows", type=int, default=20_000)
    ap.add_argument("--threads", default="16,64,256")
    ap.add_argument("--calls", type=int, default=8192)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import pyrope_b200 as pg
    from pyrope_b200 import vector_index as vi
    L = pg.load()
    pg._lib.check(L.pyrope_gpu_init(0))
    n = C.c_int32(0)
    pg._lib.check(L.pyrope_gpu_device_count(C.byref(n)))
    threads = [int(x) for x in args.threads.split(",")]
    res = {"workload": {"index": "string-id Head+Tail, IVF_PQ tail", "rows": args.rows, "head_rows": args.head_rows,
                        "dim": 128, "nlist": 4096, "m": 16, "k": 256, "nprobe": 64, "topk_mix": MIX,
                        "calls_per_arm": args.calls, "rounds": args.rounds},
           **gpu_info()}
    t0 = time.perf_counter()
    d = build_index(vi, args.rows, args.head_rows, 1)
    res["build_s"] = round(time.perf_counter() - t0, 1)
    res["n1"] = measure(vi, d, threads, args.calls, args.rounds)
    d.close()
    if n.value > 1:  # the tail sharded over every GPU of the box
        d = build_index(vi, args.rows, args.head_rows, n.value)
        res[f"n{n.value}"] = measure(vi, d, [64], args.calls, 1)
        d.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
