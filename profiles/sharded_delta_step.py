"""What a Head+Tail over a sharded tail costs on top of the sharded search itself.

At N = 1, 2, 4, 8 devices (those the box has) it builds the C5 shape (IVF_PQ, dim 128, m 16, k 256, nprobe 64, nlist
65,536 per 100 M rows, 10,000-query batch, TOPK 10) over --rows rows and times one batch, queries and results resident on
the first device, three ways:
  (a) pyrope_sharded_search_batch_device on the sharded index alone,
  (b) pyrope_delta_search_batch_device of a Head+Tail over it (pyrope_delta_create_sharded) with an empty FLAT head,
  (c) the same Head+Tail with a --head-rows FLAT head,
and, to read (c) against, (h) the head's FLAT search of the same batch alone.  Every call returns after its last device
work finished, so a host clock around each call is its step time; the sharded search's own CUDA-event time of the first
device is reported beside (a).  Warm-up calls first, then --steps timed calls per variant, interleaved.  (b) must return
exactly what (a) returns.  Prints one JSON line with the card name and power limit.

    python profiles/sharded_delta_step.py [--rows 100000000] [--head-rows 100000] [--steps 20] [--warmup 3] [--out F]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clk = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk, "gpus_visible": len(out)}
    except Exception as e:  # the numbers stay meaningful with the name torch reports
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": None, "note": f"nvidia-smi unavailable: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--head-rows", type=int, default=100_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--devices", default="1,2,4,8", help="device counts to run (those above the box's count are skipped)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import pyrope_b200 as pg
    from pyrope_b200 import _lib
    L = pg.load()
    dim, m, k, nq, topk, nprobe = 128, 16, 256, 10_000, 10, 64
    nlist = max(64, int(round(65536 * args.rows / 100_000_000)))
    ndev = torch.cuda.device_count()
    counts = [int(c) for c in args.devices.split(",") if int(c) <= ndev]
    if not counts:
        raise SystemExit("no GPU: this script measures on the device and has no CPU fallback")
    _lib.check(L.pyrope_gpu_init(0))
    torch.cuda.set_device(0)
    Q = torch.empty((nq, dim), dtype=torch.float32, device="cuda:0")
    _lib.fill_uniform_device(Q.data_ptr(), Q.numel(), 1337, 0, stream=torch.cuda.current_stream().cuda_stream)
    outs = {v: (torch.empty((nq, topk), dtype=torch.float32, device="cuda:0"),
                torch.empty((nq, topk), dtype=torch.int64, device="cuda:0"),
                torch.empty((nq,), dtype=torch.int32, device="cuda:0")) for v in "abch"}
    rng = np.random.default_rng(7)
    head_X = rng.random((args.head_rows, dim), dtype=np.float32)
    head_labels = np.arange(args.rows, args.rows + args.head_rows, dtype=np.int64)  # ids the tail does not hold
    torch.cuda.synchronize()
    results = []
    for N in counts:
        sx = pg.ShardedIndex(N, pg.IVF_PQ, dim, pg.L2, nlist=nlist, m=m, k=k)
        sx.set_train_params(min(args.rows, max(40 * nlist, 65536)), 4 if nlist > 1024 else 10)
        t0 = time.time()
        chunk = min(args.rows, (1 << 31) // (dim * 4) // 2)
        for r in range(N):  # device-resident feed, as bench.py --sharded-entry: every shard sees every row
            shard, dev = sx.shard(r)
            torch.cuda.set_device(dev)
            _lib.check(L.pyrope_gpu_init(dev))
            shard.reserve(args.rows)
            stage = torch.empty(chunk * dim, dtype=torch.float32, device=f"cuda:{dev}")
            row = 0
            while row < args.rows:
                c = min(chunk, args.rows - row)
                _lib.fill_uniform_device(stage.data_ptr(), c * dim, 42, row * dim, stream=torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
                shard.add_device(stage.data_ptr(), c)
                row += c
            del stage
            torch.cuda.empty_cache()
        sx.note_rows(args.rows)
        sx.build()
        build_s = time.time() - t0
        torch.cuda.set_device(0)
        _lib.check(L.pyrope_gpu_init(0))
        empty = pg.GpuIndex(pg.FLAT, dim, pg.L2)
        full = pg.GpuIndex(pg.FLAT, dim, pg.L2)
        full.add(head_X, labels=head_labels)
        deltas = {}
        for v, head in (("b", empty), ("c", full)):
            d = _lib.vp()
            _lib.check(L.pyrope_delta_create_sharded(head._h, sx._s, C.byref(d)))
            deltas[v] = d

        def call(v):
            sc, rw, cn = outs[v]
            if v == "a":
                sx.search_device(Q.data_ptr(), nq, topk, sc.data_ptr(), rw.data_ptr(), cn.data_ptr(), nprobe=nprobe)
            elif v == "h":
                full.search_device(Q.data_ptr(), nq, topk, sc.data_ptr(), rw.data_ptr(), cn.data_ptr(), nprobe=nprobe)
                torch.cuda.synchronize()
            else:
                _lib.check(L.pyrope_delta_search_batch_device(deltas[v], nq, _lib.vp(Q.data_ptr()), topk, -1, nprobe,
                                                              _lib.vp(sc.data_ptr()), _lib.vp(rw.data_ptr()),
                                                              _lib.vp(cn.data_ptr()), None))

        for _ in range(args.warmup):
            for v in "abch":
                call(v)
        ms = {v: [] for v in "abch"}
        dev_ms = []
        for _ in range(args.steps):  # interleaved, so drift on the shared host hits every variant alike
            for v in "abch":
                t = time.perf_counter()
                call(v)
                ms[v].append((time.perf_counter() - t) * 1e3)
                if v == "a":
                    dev_ms.append(sx.last_search_ms())
        same = all(torch.equal(outs["a"][i], outs["b"][i]) for i in range(3))
        row = {"n_gpus": N, "rows": args.rows, "nlist": nlist, "build_s": round(build_s, 1), "empty_head_equals_tail": same}
        for v, name in (("a", "sharded_ms"), ("b", "delta_empty_head_ms"), ("c", "delta_head_ms"), ("h", "head_alone_ms")):
            row[name] = {"median": round(statistics.median(ms[v]), 4), "min": round(min(ms[v]), 4),
                         "max": round(max(ms[v]), 4)}
        row["sharded_device_event_ms_median"] = round(statistics.median(dev_ms), 4)
        row["delta_overhead_empty_head_ms"] = round(row["delta_empty_head_ms"]["median"] - row["sharded_ms"]["median"], 4)
        row["delta_overhead_head_ms"] = round(row["delta_head_ms"]["median"] - row["sharded_ms"]["median"], 4)
        results.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        for d in deltas.values():
            L.pyrope_delta_destroy(d)
        empty.close()
        full.close()
        sx.close()
        torch.cuda.empty_cache()
    line = {"what": "Head+Tail over a sharded IVF_PQ tail vs the sharded search alone (one 10k-query batch, C5 shape)",
            **gpu_info(), "head_rows": args.head_rows, "nq": nq, "topk": topk, "nprobe": nprobe, "m": m, "k": k, "dim": dim,
            "steps": args.steps, "warmup": args.warmup, "timing": "host clock around calls that return after their device work",
            "results": results}
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
