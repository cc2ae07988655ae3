"""What Extend costs at the C5 shape, and what it buys the search.

Builds the C5 shape on one device (IVF_PQ, dim 128, m 16, k 256, nlist 65,536 per 100 M rows, the training bounds of
bench.py's C5 build) over --rows rows, then adds --buffer rows to the write buffer and measures, as medians of
interleaved repeats (host clock around calls that return after their device work):
  * search_buffer_ms   one 10,000-query batch (TOPK 10, nprobe 64), queries and results on the device, buffer in place;
  * search_extended_ms the same batch after Extend has moved the buffer into the lists;
  * extend_ms          pyrope_index_extend of --buffer rows (assign + encode + group + list merge), one per repeat, each
                       repeat first adding a fresh --buffer rows (so the lists grow by --buffer per repeat);
  * build_s            the full Build of the same index (--rows + --buffer rows), timed once;
  * merge kernel       extend_merge_lists_kernel's device time from torch.profiler in a separate Extend, with the
                       algorithmic bytes it moves (one read and one write of every list array, plus the new rows) and the
                       rate against an HBM copy (torch copy_ of 2 x 2 GiB) measured in the same run;
  * the dominant search kernel's name after Extend (pyrope_index_last_search_kernel), and max_list_len-dependent path.
Prints one JSON line with the card's name and power limit.

    python profiles/extend_step.py [--rows 100000000] [--buffer 1000000] [--repeats 5] [--out F]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from profiles.sharded_delta_step import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--buffer", type=int, default=1_000_000)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--search-steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import pyrope_b200 as pg
    from pyrope_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this script measures on the device and has no CPU fallback")
    L = pg.load()
    dim, m, k, nq, topk, nprobe = 128, 16, 256, 10_000, 10, 64
    nlist = max(64, int(round(65536 * args.rows / 100_000_000)))
    _lib.check(L.pyrope_gpu_init(0))
    torch.cuda.set_device(0)
    st = torch.cuda.current_stream().cuda_stream
    Q = torch.empty((nq, dim), dtype=torch.float32, device="cuda:0")
    _lib.fill_uniform_device(Q.data_ptr(), Q.numel(), 1337, 0, stream=st)
    sc = torch.empty((nq, topk), dtype=torch.float32, device="cuda:0")
    rw = torch.empty((nq, topk), dtype=torch.int64, device="cuda:0")
    cn = torch.empty((nq,), dtype=torch.int32, device="cuda:0")
    chunk = min(args.rows, (1 << 31) // (dim * 4) // 2)
    stage = torch.empty(chunk * dim, dtype=torch.float32, device="cuda:0")
    fed = [0]  # rows of the uniform stream fed so far (every row is a distinct slice of it)

    def feed(g, n):
        row = 0
        while row < n:
            c = min(chunk, n - row)
            _lib.fill_uniform_device(stage.data_ptr(), c * dim, 42, fed[0] * dim, stream=st)
            torch.cuda.synchronize()
            g.add_device(stage.data_ptr(), c)
            row += c
            fed[0] += c

    def make():
        g = pg.GpuIndex(pg.IVF_PQ, dim, pg.L2, nlist=nlist, m=m, k=k)
        g.set_train_params(min(args.rows, max(40 * nlist, 65536)), 4 if nlist > 1024 else 10)
        g.reserve(args.rows + args.buffer)
        return g

    def search(g):
        t = time.perf_counter()
        g.search_device(Q.data_ptr(), nq, topk, sc.data_ptr(), rw.data_ptr(), cn.data_ptr(), nprobe=nprobe)
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3

    # the full Build the Extend is measured against: --rows + --buffer rows in the buffer, one Build
    g = make()
    feed(g, args.rows + args.buffer)
    t = time.perf_counter()
    g.build()
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t
    g.close()
    torch.cuda.empty_cache()

    fed[0] = 0
    g = make()
    feed(g, args.rows)
    g.build()
    torch.cuda.synchronize()
    search(g)  # warm-up of the list-major path

    # copy rate of the card in this run: 2 GiB read + 2 GiB written per copy_
    a = torch.empty(1 << 29, dtype=torch.float32, device="cuda:0")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cms = []
    for _ in range(10):
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        cms.append(e0.elapsed_time(e1))
    copy_gbs = 2 * a.numel() * 4 / (statistics.median(cms) * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()

    s_buf, s_ext, ext_ms, kernels = [], [], [], []
    for rep in range(args.repeats):  # interleaved: buffer in place -> Extend -> extended
        feed(g, args.buffer)
        search(g)
        s_buf.append(statistics.median([search(g) for _ in range(args.search_steps)]))
        t = time.perf_counter()
        g.extend()
        torch.cuda.synchronize()
        ext_ms.append((time.perf_counter() - t) * 1e3)
        search(g)
        s_ext.append(statistics.median([search(g) for _ in range(args.search_steps)]))
        kernels.append(g.last_search_kernel()[0])

    # the merge kernel alone, in a profiled Extend of its own
    feed(g, args.buffer)
    tot = _lib.C.c_int64(0)
    _lib.check(L.pyrope_index_get_lists(g._h, None, None, None, _lib.C.byref(tot)))
    old_total = tot.value
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        g.extend()
        torch.cuda.synchronize()
    merge_us = sum(e.device_time_total for e in prof.key_averages() if "extend_merge_lists_kernel" in e.key)
    per_kernel = sorted(((e.key, round(e.device_time_total / 1e3, 3)) for e in prof.key_averages() if e.device_time_total > 0),
                        key=lambda x: -x[1])[:8]
    entry = m + 8 + 8  # code, row ordinal, label (no dead flags: nothing was deleted)
    merge_bytes = old_total * entry + (old_total + args.buffer) * entry + args.buffer * (entry + 4)
    merge_gbs = merge_bytes / (merge_us * 1e-6) / 1e9 if merge_us else None

    line = {"what": "Extend of a C5 IVF_PQ index on one device: search with the buffer vs after Extend, Extend vs Build",
            **gpu_info(), "rows": args.rows, "buffer_rows": args.buffer, "nlist": nlist, "m": m, "k": k, "dim": dim,
            "nq": nq, "topk": topk, "nprobe": nprobe, "repeats": args.repeats,
            "search_buffer_ms_median": round(statistics.median(s_buf), 3),
            "search_extended_ms_median": round(statistics.median(s_ext), 3),
            "search_buffer_ms": [round(x, 3) for x in s_buf], "search_extended_ms": [round(x, 3) for x in s_ext],
            "extend_ms_median": round(statistics.median(ext_ms), 1), "extend_ms": [round(x, 1) for x in ext_ms],
            "build_s": round(build_s, 2), "build_note": "one full Build of rows + buffer rows, timed once",
            "merge_kernel_ms": round(merge_us / 1e3, 3), "merge_bytes": merge_bytes,
            "merge_gbs": round(merge_gbs, 1) if merge_gbs else None,
            "copy_gbs_measured": round(copy_gbs, 1),
            "merge_share_of_copy": round(merge_gbs / copy_gbs, 3) if merge_gbs else None,
            "profiled_extend_kernels_ms": per_kernel,
            "dominant_search_kernel_after_extend": kernels,
            "timing": "host clock around calls that return after their device work; merge kernel by torch.profiler"}
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
