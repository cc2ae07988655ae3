#!/usr/bin/env python
"""bench.py — batched VEC.SEARCH throughput of the B200 hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c5|c4|c1|c2|c3|c2x] [--scale S]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the CPU arm (oracle port of the reference's C# loops)
    python bench.py ... --dump-outputs DIR    # also write the last timed step's results as DIR/<workload>_*.npy

A step = one pass of the hot path over one batch of synthetic queries.  `value` = whole-job QPS with
queries and outputs resident in HBM (CUDA events on the launching stream, max over ranks);
`e2e` = the same through the C-ABI host entry point with HOST buffers (H2D of the queries and D2H of
the results inside the timed region).  One JSON line on stdout (rank 0).

The default run measures BASELINE config 5 (IVF_PQ, the configuration the metric is quoted on) as the line
itself and BASELINE config 4 (FLAT inner product on the tensor cores) as its `secondary` block.  Every
block carries `parity`: the GPU result of the timed configuration compared with the CPU oracle (tests/parity.py
rules: scores within 1e-4 relative, ids identical except across near-ties); a mismatch exits non-zero.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC_NAME = "batched VEC.SEARCH QPS at fixed recall@10"
RTOL = 1e-4  # north_star: distances within 1e-4 relative


def workload(name: str, scale: float) -> dict:
    """BASELINE.json configs (SURVEY.md §8d).  scale < 1 shrinks N and nlist together (list length,
    nprobe and per-query work unchanged) for development runs; such lines carry "reduced": true."""
    if name == "c5":
        w = dict(kind="IVF_PQ", metric="L2", dim=128, n=100_000_000, nq=10_000, topk=10, nlist=65536, m=16, k=256,
                 nprobe=64)
        w["n"] = max(4096, int(round(w["n"] * scale)))
        w["nlist"] = max(64, int(round(w["nlist"] * scale)))
    elif name in ("c5m8", "c5m4"):  # C5's shape with fewer, longer sub-vectors (not BASELINE configs: the widened list-major scan)
        w = dict(kind="IVF_PQ", metric="L2", dim=128, n=100_000_000, nq=10_000, topk=10, nlist=65536, m=int(name[3:]), k=256,
                 nprobe=64)
        w["n"] = max(4096, int(round(w["n"] * scale)))
        w["nlist"] = max(64, int(round(w["nlist"] * scale)))
    elif name == "c4":
        w = dict(kind="FLAT", metric="IP", dim=768, n=10_000_000, nq=10_000, topk=100)
        w["n"] = max(4096, int(round(w["n"] * scale)))
    elif name == "c1":
        w = dict(kind="FLAT", metric="L2", dim=128, n=10_000, nq=100, topk=10)
    elif name == "c2x":  # IVF_FLAT at a size where the list scan is HBM/L2-bound (not a BASELINE config; roofline of K4)
        w = dict(kind="IVF_FLAT", metric="L2", dim=128, n=10_000_000, nq=10_000, topk=10, nlist=4096, nprobe=16)
        w["n"] = max(4096, int(round(w["n"] * scale)))
        w["nlist"] = max(64, int(round(w["nlist"] * scale)))
    elif name == "c2w":  # the same with rows of 768 floats (the wide list-major kernels)
        w = dict(kind="IVF_FLAT", metric="L2", dim=768, n=2_000_000, nq=10_000, topk=10, nlist=1024, nprobe=16)
        w["n"] = max(4096, int(round(w["n"] * scale)))
        w["nlist"] = max(64, int(round(w["nlist"] * scale)))
    elif name == "c2":
        w = dict(kind="IVF_FLAT", metric="L2", dim=128, n=10_000, nq=100, topk=10, nlist=100, nprobe=3)
    elif name == "c3":
        w = dict(kind="IVF_PQ", metric="L2", dim=128, n=10_000, nq=100, topk=10, nlist=100, m=4, k=256, nprobe=1)
    else:
        raise SystemExit(f"unknown workload {name}")
    w["name"] = name
    w["reduced"] = bool(scale != 1.0 and name in ("c4", "c5", "c2x", "c2w", "c5m8", "c5m4"))
    return w


def describe(w: dict) -> str:
    if w["kind"] == "IVF_PQ":
        return (f"{w['name']}: IVF_PQ nlist={w['nlist']} m={w['m']} k={w['k']} synthetic dim={w['dim']}, "
                f"{w['n']} base, nprobe={w['nprobe']}, {w['nq']}-query batch, TOPK {w['topk']}")
    if w["kind"] == "IVF_FLAT":
        return (f"{w['name']}: IVF_FLAT nlist={w['nlist']} synthetic dim={w['dim']}, {w['n']} base, "
                f"nprobe={w['nprobe']}, {w['nq']} queries, TOPK {w['topk']}")
    return f"{w['name']}: FLAT {w['metric']} synthetic dim={w['dim']}, {w['n']} base, {w['nq']}-query batch, TOPK {w['topk']}"


def config_of(w: dict) -> dict:
    """The `config` object: identical in the GPU arm and the reference arm (everything else lives in `details`)."""
    return {"workload": describe(w), "reduced": w["reduced"]}


def dtype_of(w: dict) -> str:
    return "f32" if w["kind"] != "IVF_PQ" else "f32 LUT / u8 codes"


def algorithmic_work(w: dict, world: int) -> dict:
    """Per search launch on ONE rank (SURVEY.md §8d): HBM bytes for the scan paths, FLOPs for FLAT."""
    if w["kind"] == "IVF_PQ":  # codes only: nprobe * avg_list * m bytes per query
        b = w["nq"] * w["nprobe"] * (w["n"] / w["nlist"]) * w["m"] / world
        return {"bound": "hbm", "work": b, "unit": "GB/s"}
    if w["kind"] == "IVF_FLAT":
        b = w["nq"] * (w["nprobe"] * (w["n"] / w["nlist"]) * w["dim"] * 4) / world
        return {"bound": "hbm", "work": b, "unit": "GB/s"}
    f = 2.0 * w["nq"] * (w["n"] / world) * w["dim"]
    return {"bound": "tensor", "work": f, "unit": "TFLOP/s"}


def host_cores() -> int:
    """Cores this process may run on.  (torchrun exports OMP_NUM_THREADS=1, so omp_get_max_threads() is not it.)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def log(s):
    print(s, file=sys.stderr, flush=True)


def dump_outputs(out_dir, name: str, scores, ids, counts):
    """--dump-outputs: what a caller of the timed search receives from its last step, as out_dir/<name>_scores.npy
    (float32 [nq][k]), <name>_ids.npy and <name>_counts.npy (float64: exact for ids below 2**53), so that two builds
    can be compared on the same seeded inputs.  nq <= 10,000 and k <= 100 in every workload: at most 13 MB per workload."""
    if not out_dir:
        return
    os.makedirs(out_dir, exist_ok=True)
    for part, a, dt in (("scores", scores, np.float32), ("ids", ids, np.float64), ("counts", counts, np.float64)):
        np.save(os.path.join(out_dir, f"{name}_{part}.npy"), np.asarray(a).astype(dt))


# ------------------------------------------------------------------------------------------------
# index construction on the GPU (setup, untimed)
# ------------------------------------------------------------------------------------------------
def build_gpu_index(pg, torch, w: dict, rank: int, world: int):
    from pyrope_b200 import _lib
    kind = {"FLAT": pg.FLAT, "IVF_FLAT": pg.IVF_FLAT, "IVF_PQ": pg.IVF_PQ}[w["kind"]]
    metric = {"L2": pg.L2, "IP": pg.INNER_PRODUCT, "COSINE": pg.COSINE}[w["metric"]]
    dim, n = w["dim"], w["n"]
    ix = pg.GpuIndex(kind, dim, metric, nlist=w.get("nlist", 100), m=w.get("m", 4), k=w.get("k", 256))
    t0 = time.time()
    if kind == pg.FLAT:
        from pyrope_b200.shard import row_block
        lo, hi = row_block(n, rank, world)  # contiguous row blocks per rank
    else:
        lo, hi = 0, n  # every rank sees every row; lists are sharded by list id at build time
        if world > 1:
            ix.set_shard(rank, world)
        ntrain = min(n, max(40 * w["nlist"], 65536))
        ix.set_train_params(ntrain, 4 if w["nlist"] > 1024 else 10)
    ix.reserve(hi - lo)
    chunk = min(hi - lo, (1 << 31) // (dim * 4) // 2)  # ~1 GiB staging
    stage = torch.empty(chunk * dim, dtype=torch.float32, device="cuda")
    labels = torch.empty(chunk, dtype=torch.int64, device="cuda") if kind == pg.FLAT and world > 1 else None
    r = lo
    while r < hi:
        c = min(chunk, hi - r)
        _lib.fill_uniform_device(stage.data_ptr(), c * dim, 42, r * dim, stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        if labels is not None:
            labels[:c] = torch.arange(r, r + c, device="cuda")
            ix.add_device(stage.data_ptr(), c, labels.data_ptr())
        else:
            ix.add_device(stage.data_ptr(), c)
        r += c
    del stage
    t1 = time.time()
    if kind != pg.FLAT:
        ix.build()
    t2 = time.time()
    log(f"rank {rank}: {w['name']}: added {hi - lo} rows in {t1 - t0:.1f}s, build {t2 - t1:.1f}s, stats {ix.stats()}")
    return ix, {"add_s": round(t1 - t0, 2), "build_s": round(t2 - t1, 2)}


def make_queries(torch, w: dict):
    from pyrope_b200 import _lib
    q = torch.empty(w["nq"] * w["dim"], dtype=torch.float32, device="cuda")
    _lib.fill_uniform_device(q.data_ptr(), q.numel(), 1337, 0, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return q.view(w["nq"], w["dim"])


def recall_at_10(pg, torch, w: dict, ix, Q, nq_eval: int) -> dict:
    """recall@10 of the configured index against exact FLAT top-10 (SURVEY.md §8d: the reference never computes
    recall; the metric is quoted 'at fixed recall@10', i.e. at the recall this (nlist, nprobe, m) gives).
    Exact answers: the base is regenerated chunk by chunk into a FLAT index on the CUDA-core path (no split
    copies), per-chunk top-10 lists are merged with pyrope_topk_merge_device.  Setup work, untimed."""
    from pyrope_b200 import _lib
    k = 10
    nq_eval = min(nq_eval, w["nq"])
    metric = {"L2": pg.L2, "IP": pg.INNER_PRODUCT, "COSINE": pg.COSINE}[w["metric"]]
    dim, n = w["dim"], w["n"]
    q = Q[:nq_eval].contiguous()
    stream = torch.cuda.current_stream().cuda_stream
    chunk = min(n, 10_000_000)
    nchunks = (n + chunk - 1) // chunk
    S = torch.zeros((nchunks, nq_eval, k), dtype=torch.float32, device="cuda")
    R = torch.full((nchunks, nq_eval, k), -1, dtype=torch.int64, device="cuda")
    cnt = torch.empty((nq_eval,), dtype=torch.int32, device="cuda")
    stage = torch.empty(chunk * dim, dtype=torch.float32, device="cuda")
    labels = torch.empty(chunk, dtype=torch.int64, device="cuda")
    old = os.environ.get("PYROPE_FLAT_TC")
    os.environ["PYROPE_FLAT_TC"] = "0"
    try:
        for c in range(nchunks):
            r0 = c * chunk
            rows = min(chunk, n - r0)
            _lib.fill_uniform_device(stage.data_ptr(), rows * dim, 42, r0 * dim, stream=stream)
            labels[:rows] = torch.arange(r0, r0 + rows, device="cuda")
            torch.cuda.synchronize()
            fx = pg.GpuIndex(pg.FLAT, dim, metric)
            fx.add_device(stage.data_ptr(), rows, labels.data_ptr())
            fx.search_device(q.data_ptr(), nq_eval, k, S[c].data_ptr(), R[c].data_ptr(), cnt.data_ptr(), stream=stream)
            torch.cuda.synchronize()
            fx.close()
    finally:
        if old is None:
            os.environ.pop("PYROPE_FLAT_TC", None)
        else:
            os.environ["PYROPE_FLAT_TC"] = old
    ms = torch.empty((nq_eval, k), dtype=torch.float32, device="cuda")
    mr = torch.empty((nq_eval, k), dtype=torch.int64, device="cuda")
    _lib.topk_merge_device(nq_eval, nchunks, k, k, S.data_ptr(), R.data_ptr(), ms.data_ptr(), mr.data_ptr(), cnt.data_ptr(),
                           stream=stream)
    gs = torch.empty((nq_eval, k), dtype=torch.float32, device="cuda")
    gr = torch.empty((nq_eval, k), dtype=torch.int64, device="cuda")
    ix.search_device(q.data_ptr(), nq_eval, k, gs.data_ptr(), gr.data_ptr(), cnt.data_ptr(), nprobe=w.get("nprobe", -1), stream=stream)
    torch.cuda.synchronize()
    truth, got = mr.cpu().numpy(), gr.cpu().numpy()
    hit = sum(len(set(t.tolist()) & set(g.tolist()) - {-1}) for t, g in zip(truth, got))
    del stage, labels, S, R
    torch.cuda.empty_cache()
    return {"recall_at_10": round(hit / (nq_eval * k), 4), "recall_queries": nq_eval,
            "recall_truth": "exact FLAT top-10 over the full base (GPU CUDA-core path, chunked)"}


# ------------------------------------------------------------------------------------------------
# parity: the GPU result of the timed configuration against the CPU oracle (tests/parity.py rules)
# ------------------------------------------------------------------------------------------------
def compare_topk(ref, got, what: str) -> dict:
    """ref / got = (ids [nq][k], scores [nq][k], counts [nq]) for the same queries.  Counts mismatching queries by the
    rules of tests/parity.py (scores within RTOL relative; id lists identical except where the reference's own scores
    are within tolerance of each other, or of its k-th score at the boundary) and reports the worst relative score error."""
    from tests.parity import assert_topk_equivalent
    rid, rsc, rcn = ref
    gid, gsc, gcn = got
    nq = len(rcn)
    mismatch, first, max_rel, exact_ids = 0, None, 0.0, 0
    for q in range(nq):
        c = int(rcn[q])
        try:
            if int(gcn[q]) != c:
                raise AssertionError(f"count {int(gcn[q])} != reference {c}")
            assert_topk_equivalent(rid[q][:c], rsc[q][:c], gid[q][:c], gsc[q][:c], rtol=RTOL, ctx=f"q{q}")
        except AssertionError as ex:
            mismatch += 1
            if first is None:
                first = str(ex)[:300]
            continue
        if c:
            a, b = np.asarray(rsc[q][:c], np.float64), np.asarray(gsc[q][:c], np.float64)
            den = np.maximum(np.maximum(np.abs(a), np.abs(b)), 1e-30)
            max_rel = max(max_rel, float(np.max(np.abs(a - b) / den)))
            exact_ids += int(np.array_equal(np.asarray(rid[q][:c]), np.asarray(gid[q][:c])))
    out = {"queries": nq, "mismatch": mismatch, "max_rel_err": max_rel, "identical_id_lists": exact_ids, "rtol": RTOL,
           "against": what}
    if first:
        out["first_mismatch"] = first
    return out


def base_rows_host(torch, w: dict, n_rows: int) -> np.ndarray:
    """The first n_rows base vectors, regenerated with the same counter-based generator."""
    from pyrope_b200 import _lib
    t = torch.empty(n_rows * w["dim"], dtype=torch.float32, device="cuda")
    _lib.fill_uniform_device(t.data_ptr(), t.numel(), 42, 0, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return t.view(n_rows, w["dim"]).cpu().numpy()


def oracle_index_from_gpu(ix, w: dict, torch=None):
    """-> (oracle index, rows it holds, note).  IVF_PQ adopts the GPU-built lists (same codebooks, codes);
    FLAT / IVF_FLAT are rebuilt by the oracle from (a bounded prefix of) the same synthetic rows."""
    from oracle import pyoracle as orc
    metric = {"L2": orc.L2, "IP": orc.IP, "COSINE": orc.COSINE}[w["metric"]]
    if w["kind"] == "IVF_PQ":
        o = orc.IvfPqIndex(w["dim"], metric, m=w["m"], k=w["k"], nlist=w["nlist"])
        off, rows, codes = ix.lists()
        cb, _ = ix.codebooks()
        o.adopt(ix.centroids(), cb, off, rows, codes)
        return o, w["n"], "the GPU-built index (same codebooks, lists and codes)"
    if w["kind"] == "FLAT":
        ns = min(w["n"], max(10_000, (256 << 20) // (w["dim"] * 4)))  # <= 256 MiB of rows on the host
        o = orc.FlatIndex(w["dim"], metric)
        o.add_batch(base_rows_host(torch, w, ns))
        return o, ns, f"the first {ns} of {w['n']} base rows (QPS scaled by {ns}/{w['n']}: the scan is linear in rows)"
    if w["kind"] == "IVF_FLAT" and w["n"] <= 200_000:
        o = orc.IvfFlatIndex(w["dim"], metric, nlist=w["nlist"])
        o.add_batch(base_rows_host(torch, w, w["n"]))
        o.build()
        return o, w["n"], "an oracle-built index over the same rows"
    if w["kind"] == "IVF_FLAT" and w["n"] * w["dim"] * 4 <= (12 << 30):  # the rows fit on the host twice over
        o = orc.IvfFlatIndex(w["dim"], metric, nlist=w["nlist"])
        off, rows, _ = ix.lists()
        base = base_rows_host(torch, w, w["n"])
        o.adopt(ix.centroids(), off, rows, base[rows])   # list-major copy of the same rows
        return o, w["n"], "the GPU-built index (same centroids and lists)"
    raise NotImplementedError


def _osearch(oidx, Q, w, threads):
    if w["kind"] == "FLAT":
        return oidx.search_batch(Q, w["topk"], nthreads=threads)
    return oidx.search_batch(Q, w["topk"], nprobe=w.get("nprobe", -1), nthreads=threads)


def time_cpu_baseline(oidx, rows_held, note, Qh: np.ndarray, w: dict, budget_s: float):
    """-> (cpu_baseline dict, queries searched, oracle result for them)."""
    threads = host_cores()
    probe = min(len(Qh), 2 * threads)
    t0 = time.perf_counter()
    _osearch(oidx, Qh[:probe], w, threads)
    per_q = (time.perf_counter() - t0) / probe
    s = int(max(threads, min(len(Qh), budget_s / max(per_q, 1e-9))))
    t0 = time.perf_counter()
    res = _osearch(oidx, Qh[:s], w, threads)
    dt = time.perf_counter() - t0
    scale = rows_held / w["n"]
    return {"value": round(s / dt * scale, 2), "unit": "QPS", "cores": threads, "kind": "port",
            "sample": f"{s} of the batch's {len(Qh)} queries over {note}, one query per thread, {dt:.1f}s wall"}, s, res


def flat_fullsize_parity(pg, torch, w: dict, Qh: np.ndarray, got, nsample: int) -> dict:
    """FLAT at a size the CPU oracle cannot scan (C4: 30.7 GB per query): for a sample of the batch's queries,
      (1) every reported score must equal — bit for bit — the oracle's VectorMath.DotProductUnsafe / L2SquaredUnsafe
          of that query and that row (rows regenerated on the host from the counter-based generator);
      (2) the id list must agree (tests/parity.py rules) with an INDEPENDENT exact top-k over the whole regenerated base
          (fp32 cuBLAS SGEMM, TF32 off, chunk by chunk, + torch.topk: library code used only as a checker)."""
    from oracle import pyoracle as orc
    from pyrope_b200 import _lib
    dim, n, k = w["dim"], w["n"], w["topk"]
    ns = min(nsample, len(Qh))
    gsc, gid, gcn = got
    stream = torch.cuda.current_stream().cuda_stream
    old_tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        Qs = torch.from_numpy(np.ascontiguousarray(Qh[:ns])).cuda()
        chunk = min(n, 2_000_000)
        stage = torch.empty(chunk * dim, dtype=torch.float32, device="cuda")
        best_s, best_i = None, None
        for r0 in range(0, n, chunk):
            rows = min(chunk, n - r0)
            _lib.fill_uniform_device(stage.data_ptr(), rows * dim, 42, r0 * dim, stream=stream)
            X = stage[:rows * dim].view(rows, dim)
            if w["metric"] == "IP":
                S = Qs @ X.T
            else:
                S = 2.0 * (Qs @ X.T) - (X * X).sum(1)[None, :] - (Qs * Qs).sum(1)[:, None]
            s, i = torch.topk(S, min(k, rows), dim=1)
            i = i + r0
            if best_s is None:
                best_s, best_i = s, i
            else:
                cs, ci = torch.cat([best_s, s], 1), torch.cat([best_i, i], 1)
                s2, j = torch.topk(cs, min(k, cs.shape[1]), dim=1)
                best_s, best_i = s2, torch.gather(ci, 1, j)
            del S
        ref_ids = best_i.cpu().numpy()
        # (1) + reference scores for (2): oracle arithmetic on the union of the ids either side reports
        rowbuf = torch.empty(dim, dtype=torch.float32, device="cuda")
        cache = {}

        def row(r):
            if r not in cache:
                _lib.fill_uniform_device(rowbuf.data_ptr(), dim, 42, int(r) * dim, stream=stream)
                torch.cuda.synchronize()
                cache[r] = rowbuf.cpu().numpy().copy()
            return cache[r]

        f = orc.dot_unsafe if w["metric"] == "IP" else (lambda a, b: -orc.l2sq_unsafe(a, b))
        bit_exact, checked = 0, 0
        ref_sc = np.zeros((ns, k), np.float32)
        for q in range(ns):
            for j in range(int(gcn[q])):
                s_or = np.float32(f(Qh[q], row(int(gid[q][j]))))
                checked += 1
                bit_exact += int(s_or == np.float32(gsc[q][j]))
            sc = np.array([np.float32(f(Qh[q], row(int(r)))) for r in ref_ids[q]], np.float32)
            order = np.argsort(-sc, kind="stable")
            ref_ids[q] = ref_ids[q][order]
            ref_sc[q] = sc[order]
            cache.clear()
        cnt = np.full(ns, min(k, n), np.int32)
        out = compare_topk((ref_ids, ref_sc, cnt), (gid[:ns], gsc[:ns], gcn[:ns]),
                           "independent exact top-k over the whole base (fp32 SGEMM + topk), scored in the oracle's "
                           "VectorMath arithmetic")
        out["scores_bit_exact_vs_oracle"] = f"{bit_exact}/{checked}"
        if bit_exact != checked:
            out["mismatch"] += 1
            out.setdefault("first_mismatch", "a reported score differs from the oracle's arithmetic on the same row")
        return out
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old_tf32


def tf32_peak(torch) -> dict:
    """Dense TF32 tensor-pipe peak as cuBLAS reaches it (fp32 inputs, TF32 allowed, 8192^3): the denominator of the FLAT
    roofline.  Read from profiles/tf32_peak.json when committed, measured live (best of 10, ~1.5 ms each) otherwise."""
    path = os.path.join(ROOT, "profiles", "tf32_peak.json")
    try:
        d = json.load(open(path))
        if d.get("tf32_tflops"):
            return {"tflops": float(d["tf32_tflops"]), "source": "profiles/tf32_peak.json (cuBLAS TF32 8192^3, measured burst)"}
    except Exception:
        pass
    try:
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        n = 8192
        a = torch.randn(n, n, device="cuda")
        b = torch.randn(n, n, device="cuda")
        for _ in range(3):
            a @ b
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        torch.backends.cuda.matmul.allow_tf32 = old
        del a, b
        torch.cuda.empty_cache()
        return {"tflops": 2.0 * n ** 3 / (best / 1e3) / 1e12, "source": "cuBLAS TF32 8192^3 measured in this run (best of 10)"}
    except Exception as ex:
        return {"tflops": None, "source": f"unmeasured ({str(ex)[:80]})"}


# ------------------------------------------------------------------------------------------------
def bench_workload(args, torch, pg, dist, w: dict, steps: int, warmup: int, rank: int, world: int, local: int) -> dict:
    """Build the index of workload w, time `steps` search steps, and return the bench line (rank 0; None elsewhere)."""
    from pyrope_b200 import _lib
    nq, dim, k = w["nq"], w["dim"], w["topk"]
    nprobe = w.get("nprobe", -1)

    ix, build_info = build_gpu_index(pg, torch, w, rank, world)
    Q = make_queries(torch, w)
    stream = torch.cuda.current_stream().cuda_stream
    sc = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    rw = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    cn = torch.empty((nq,), dtype=torch.int32, device="cuda")
    if world > 1:
        g_sc = torch.empty((world, nq, k), dtype=torch.float32, device="cuda")
        g_rw = torch.empty((world, nq, k), dtype=torch.int64, device="cuda")
        m_sc, m_rw, m_cn = torch.empty_like(sc), torch.empty_like(rw), torch.empty_like(cn)
    else:
        m_sc, m_rw, m_cn = sc, rw, cn

    launches = [0]

    split_coarse = world > 1 and w["kind"] != "FLAT"
    if split_coarse:  # every rank ranks centroids for its slice of the batch; probe lists are all-gathered
        from pyrope_b200.shard import query_slice
        qlo, qhi, per = query_slice(nq, rank, world)
        P_eff = nprobe if nprobe > 0 else (3 if w["kind"] == "IVF_FLAT" else 1)
        pr_local = torch.full((per, P_eff), -1, dtype=torch.int64, device="cuda")
        pr_all = torch.empty((world * per, P_eff), dtype=torch.int64, device="cuda")

    # the step's all-gathers: peer stores over NVLink through the library (csrc/peer.cu) unless --nccl-exchange, or unless
    # some rank cannot map its peers' buffers (then every rank uses NCCL)
    grp = None
    if world > 1 and not args.nccl_exchange:
        pbytes = per * P_eff * 8 if split_coarse else 16
        ok = (nq * k) % 4 == 0 and pbytes % 16 == 0
        try:
            if ok:
                grp = _lib.PeerGroup(world, rank, max(pbytes, nq * k * 8), 3)
                mine = torch.frombuffer(bytearray(grp.handle()), dtype=torch.uint8).cuda()
        except Exception as ex:
            log(f"rank {rank}: peer exchange unavailable ({ex})")
            ok = False
        if not ok or grp is None:
            ok, mine = False, torch.zeros(64, dtype=torch.uint8, device="cuda")
        allh = torch.empty((world, 64), dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(allh.view(-1), mine)
        if ok:
            try:
                grp.open(bytes(allh.cpu().numpy().tobytes()))
            except Exception as ex:
                log(f"rank {rank}: peer exchange unavailable ({ex})")
                ok = False
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if not bool(flag.item()):
            if grp is not None:
                grp.close()
            grp = None
    collective = "none" if world == 1 else ("peer stores over NVLink + epoch flags (pyrope_peer_allgather_device)" if grp else "nccl all_gather")

    def step(marks=None):
        """One search step.  marks: a list that receives (phase name, CUDA event) pairs - the per-phase breakdown of the
        multi-GPU step (`step_phases_ms`), recorded outside the timed region only."""
        def mark(name):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                marks.append((name, ev))
        mark("start")
        if split_coarse:
            if qhi > qlo:
                ix.coarse_probe_device(Q[qlo:qhi].data_ptr(), qhi - qlo, P_eff, pr_local.data_ptr(), stream=stream)
            lc = ix.last_search_launches()
            mark("coarse_probe_own_queries")
            if grp is not None:
                probes_ptr = grp.allgather(0, pr_local.data_ptr(), per * P_eff * 8, stream=stream)
                lc += 2
            else:
                dist.all_gather_into_tensor(pr_all.view(-1), pr_local.view(-1))
                probes_ptr = pr_all.data_ptr()
            mark("allgather_probes")
            ix.search_probed_device(Q.data_ptr(), nq, k, P_eff, probes_ptr, sc.data_ptr(), rw.data_ptr(),
                                    cn.data_ptr(), stream=stream)
            launches[0] = lc + ix.last_search_launches()
        else:
            ix.search_device(Q.data_ptr(), nq, k, sc.data_ptr(), rw.data_ptr(), cn.data_ptr(), nprobe=nprobe, stream=stream)
            launches[0] = ix.last_search_launches()
        mark("search_own_shard")
        if world > 1:
            if grp is not None:
                gs_ptr = grp.allgather(1, sc.data_ptr(), nq * k * 4, stream=stream)
                gr_ptr = grp.allgather(2, rw.data_ptr(), nq * k * 8, stream=stream)
                launches[0] += 4
            else:
                dist.all_gather_into_tensor(g_sc.view(-1), sc.view(-1))
                dist.all_gather_into_tensor(g_rw.view(-1), rw.view(-1))
                gs_ptr, gr_ptr = g_sc.data_ptr(), g_rw.data_ptr()
            mark("allgather_results")
            _lib.topk_merge_device(nq, world, k, k, gs_ptr, gr_ptr, m_sc.data_ptr(), m_rw.data_ptr(),
                                   m_cn.data_ptr(), stream=stream)
            launches[0] += 1
            mark("merge")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    barrier()
    exchange = "none"
    if split_coarse and w["kind"] == "IVF_PQ" and not args.no_threshold_exchange:
        # share per-query thresholds between the ranks while their scan kernels run (NVLink peer memory, CUDA IPC):
        # one unshared step is kept to check that the merged result is the same with the exchange on
        # (every rank runs the same collectives whether or not its own set-up succeeds)
        ref_sc, ref_rw = m_sc.clone(), m_rw.clone()
        ok = True
        try:
            handle = ix.threshold_exchange_handle(nq)
        except Exception as ex:
            log(f"rank {rank}: threshold exchange unavailable ({ex})")
            handle, ok = bytes(64), False
        mine = torch.frombuffer(bytearray(handle), dtype=torch.uint8).cuda()
        allh = torch.empty((world, 64), dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(allh.view(-1), mine)
        if ok:
            try:
                ix.threshold_exchange_open(world, rank, bytes(allh.cpu().numpy().tobytes()))
            except Exception as ex:
                log(f"rank {rank}: threshold exchange unavailable ({ex})")
                ok = False
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        all_ok = bool(flag.item())
        barrier()
        for _ in range(2):
            step()
        barrier()
        same = bool(torch.equal(ref_rw, m_rw)) and bool(torch.equal(ref_sc, m_sc))
        log(f"rank {rank}: threshold exchange {'on' if all_ok else 'partly on'}, merged result identical to the unshared search: {same}")
        if ok and (not same or not all_ok):  # all or nothing
            ix.threshold_exchange_close()
        barrier()
        if same and all_ok:
            exchange = "in-kernel atomicMax of per-query thresholds into the peers' arrays (NVLink peer memory)"
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    value = nq * steps / (ms / 1e3)
    # the result every later check looks at: the merged output of the last timed step
    res_sc, res_rw, res_cn = m_sc.cpu().numpy(), m_rw.cpu().numpy(), m_cn.cpu().numpy()
    if rank == 0:
        dump_outputs(args.dump_outputs, w["name"], res_sc, res_rw, res_cn)

    # ---- dominant-kernel time (CUDA events inside the library around the scan stage), per launch
    stage_ms = {"total": 0.0, "coarse": 0.0, "scan": 0.0, "merge": 0.0}
    reps = max(3, min(steps, 10))
    kname, kms_avg = "", 0.0
    phases = {}
    for _ in range(reps):
        marks = []
        step(marks)
        torch.cuda.synchronize()
        for (_, e_a), (name, e_b) in zip(marks, marks[1:]):
            phases[name] = phases.get(name, 0.0) + e_a.elapsed_time(e_b) / reps
        for kk, v in ix.last_search_ms().items():  # with a split coarse stage: the probed search only
            stage_ms[kk] += v / reps
        kname, kms = ix.last_search_kernel()
        kms_avg += kms / reps
    if args.profile_step:  # `ncu --profile-from-start off`: exactly one search step lies inside the profiled range
        torch.cuda.profiler.start()
        step()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    alg = algorithmic_work(w, world)
    scanned = 0
    if w["kind"] in ("IVF_PQ", "IVF_FLAT"):
        scanned = ix.last_search_scanned()
    dom_ms = kms_avg if kms_avg > 0 else stage_ms["scan"]
    if not kname:
        kname = w["kind"].lower() + "_scan (stage)"
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    extra = {}
    work = alg["work"]
    if alg["bound"] == "hbm":
        # `achieved` uses SURVEY.md §8(d)'s per-unit figure (nprobe x average list x bytes per entry, per query) x
        # the queries of the launch.  The codes a launch really scores are counted on the device as well: queries
        # land in longer-than-average lists, and every list is re-read from L2 by the work items that share it, so
        # that second rate can exceed the HBM copy peak; it is reported beside, not as the roofline fraction.
        peak = peaks.get("hbm_gbs", 6650.0)
        if scanned > 0:
            exact = float(scanned) * (w["m"] if w["kind"] == "IVF_PQ" else w["dim"] * 4)
            extra["scanned_bytes_counted_on_device"] = exact
            extra["achieved_by_scanned_count"] = round(exact / (dom_ms / 1e3) / 1e9, 2)
            extra["frac_by_scanned_count"] = round(exact / (dom_ms / 1e3) / 1e9 / peak, 4)
        achieved = work / (dom_ms / 1e3) / 1e9
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (of fallback)"
        # the same bytes over the whole step (north_star's >= 60 % target read at step level)
        extra["step_level_frac"] = round(work * world / (ms / steps / 1e3) / 1e9 / (peak * world), 4)
    else:
        achieved = work / (dom_ms / 1e3) / 1e12
        tp = tf32_peak(torch) if rank == 0 else {"tflops": None, "source": ""}
        if tp["tflops"]:
            peak, peak_src = round(tp["tflops"], 1), tp["source"]
        else:
            peak = peaks.get("bf16_tflops", 1590.0) / 2.0
            peak_src = "bf16 cuBLAS burst / 2 (TF32 dense assumed; TF32 itself unmeasured)"
        terms = 1.0 if "1x" in kname else 3.0              # the 3xTF32 split issues three MMAs per useful one
        if "FP16" in kname and peaks.get("bf16_tflops"):   # kind::f16 runs at the bf16 rate: that is this pass's pipe peak
            peak, peak_src = round(float(peaks["bf16_tflops"]), 1), "MEASURED_PEAKS.json bf16_tflops (kind::f16 pass)"
            extra["tf32_peak"] = round(tp["tflops"], 1) if tp["tflops"] else None
        extra["mma_terms"] = int(terms)
        extra["issued"] = round(terms * achieved, 2)
        extra["issued_frac"] = round(terms * achieved / peak, 4)
    traffic, traffic_note = None, None
    try:
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        tr = json.load(open(tpath))
        ent = tr.get(f"{kname.split(' ')[0]}:{w['name']}:{args.scale:g}") if world == 1 else None
        if isinstance(ent, dict):
            traffic = ent.get("bytes")
            import hashlib
            stale = False
            for fn, digest in dict(ent.get("sources", {})).items():  # {file: sha256 prefix at capture time}
                fp = os.path.join(ROOT, "pyrope_b200", "csrc", fn)
                if os.path.exists(fp) and hashlib.sha256(open(fp, "rb").read()).hexdigest()[:16] != digest:
                    stale = True
            if stale:
                traffic_note = "profiles/traffic.json predates the kernel source: re-capture with ncu --set full"
                log("WARNING: " + traffic_note)
        elif ent is not None:
            traffic = ent
    except Exception:
        pass
    roofline = {"bound": alg["bound"], "achieved": round(achieved, 2), "peak": peak, "unit": alg["unit"],
                "frac": round(achieved / peak, 4), "traffic": traffic, "kernel": kname,
                "kernel_ms": round(dom_ms, 4), "algorithmic_per_launch": work, "peak_source": peak_src,
                "stage_ms": {a: round(b, 4) for a, b in stage_ms.items()},
                "step_phases_ms": {a: round(b, 4) for a, b in phases.items()}, **extra}
    if traffic_note:
        roofline["traffic_note"] = traffic_note

    # ---- end to end through the host entry point: pinned host queries in, host results out
    Qh_t = torch.empty((nq, dim), dtype=torch.float32, pin_memory=True)
    Qh_t.copy_(Q)
    torch.cuda.synchronize()
    Qh = Qh_t.numpy()
    hs = torch.empty((nq, k), dtype=torch.float32, pin_memory=True)
    hr = torch.empty((nq, k), dtype=torch.int64, pin_memory=True)
    hc = torch.empty((nq,), dtype=torch.int32, pin_memory=True)
    L = pg.load()
    import ctypes as C

    def e2e_step():
        if world == 1:
            _lib.check(L.pyrope_index_search_batch(ix._h, nq, C.c_void_p(Qh_t.data_ptr()), k, -1, nprobe,
                                                   C.c_void_p(hs.data_ptr()), C.c_void_p(hr.data_ptr()),
                                                   C.c_void_p(hc.data_ptr())))
        else:
            Q.copy_(Qh_t, non_blocking=True)
            step()
            hs.copy_(m_sc, non_blocking=True)
            hr.copy_(m_rw, non_blocking=True)
            hc.copy_(m_cn, non_blocking=True)
            torch.cuda.synchronize()

    for _ in range(max(1, min(warmup, 3))):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = {"value": round(nq * steps / e2e_s, 1), "unit": "QPS", "h2d_bytes_per_step": nq * dim * 4,
           "d2h_bytes_per_step": nq * k * 12 + nq * 4}
    e2e_same = bool(np.array_equal(hr.numpy(), res_rw) and np.array_equal(hs.numpy(), res_sc))

    # ---- recall@10 of this configuration (N=1, IVF workloads): what "at fixed recall@10" refers to
    recall = {}
    if world == 1 and w["kind"] != "FLAT" and args.recall_queries > 0:
        try:
            recall = recall_at_10(pg, torch, w, ix, Q, args.recall_queries)
        except Exception as ex:  # never lose the bench line over the quality read-out
            recall = {"recall_at_10": None, "recall_error": str(ex)[:200]}

    # ---- CPU baseline beside it + parity against the oracle (rank 0)
    cpu, parity = None, None
    if rank == 0 and not args.no_cpu:
        try:
            if w["kind"] == "IVF_PQ":
                if world == 1:
                    oix = ix
                else:
                    # the oracle needs every list: rank 0 builds the UNSHARDED index of the same rows once more (k-means /
                    # PQ training are bit-exact and deterministic, so its codebooks and codes equal the shards')
                    torch.cuda.empty_cache()
                    oix, _ = build_gpu_index(pg, torch, w, 0, 1)
                oidx, held, note = oracle_index_from_gpu(oix, w, torch)
                if oix is not ix:
                    oix.close()
                cpu, s, ores = time_cpu_baseline(oidx, held, note, Qh, w, args.cpu_budget)
                parity = compare_topk(ores, (res_rw[:s], res_sc[:s], res_cn[:s]),
                                      "oracle/oracle.c (IvfPqVectorIndex.Search restated) on the same index"
                                      + ("" if world == 1 else f": merged top-k of {world} GPUs vs the unsharded oracle"))
                del oidx
            elif w["kind"] == "FLAT" and w["n"] * w["dim"] * 4 > (256 << 20):
                oidx, held, note = oracle_index_from_gpu(ix, w, torch)
                cpu, _, _ = time_cpu_baseline(oidx, held, note, Qh, w, args.cpu_budget)
                cpu["sample"] += " (extrapolated to the full base)"
                del oidx
                parity = flat_fullsize_parity(pg, torch, w, Qh, (res_sc, res_rw, res_cn), args.flat_parity_queries)
            else:
                oidx, held, note = oracle_index_from_gpu(ix, w, torch)
                cpu, s, ores = time_cpu_baseline(oidx, held, note, Qh, w, args.cpu_budget)
                parity = compare_topk(ores, (res_rw[:s], res_sc[:s], res_cn[:s]), "oracle/oracle.c on the same rows")
                del oidx
        except NotImplementedError:
            cpu = {"value": None, "unit": "QPS", "cores": 0, "kind": "port", "sample": "not wired for this workload"}
        if parity is not None:
            parity["e2e_result_identical_to_device_result"] = e2e_same

    line = None
    if rank == 0:
        line = {
            "metric": METRIC_NAME, "value": round(value, 1), "unit": "QPS", "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": round(ms / steps, 4), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": dtype_of(w),
            "data": "synthetic uniform[0,1) fp32, counter-based generator (base seed 42, query seed 1337), "
                    "codebooks trained on device and frozen",
            "config": config_of(w),
            "details": {"l2_policy": "inputs larger than L2 (index "
                        f"{w['n'] * w.get('m', w['dim'] * 4) / 1e6:.0f} MB scanned region vs 126 MB L2)",
                        "parallelism": f"lists sharded list_id % {world}" if w["kind"] != "FLAT" else f"rows sharded in {world} blocks",
                        **recall, "exchange": ("all-gather of probe lists (coarse stage split by query) + " if split_coarse else "") +
                                    ("all-gather of per-rank top-k + on-device merge" if world > 1 else "none") +
                                    ("" if exchange == "none" else " + " + exchange),
                        "collective": collective, **build_info},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches[0] * steps),
            "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
        }
    if grp is not None:
        torch.cuda.synchronize()
        grp.close()
    ix.close()
    del ix
    torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
    return line


def run_ours(args):
    import torch

    import pyrope_b200 as pg
    from pyrope_b200 import _lib

    rank, world, local = dist_env()
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    _lib.check(pg.load().pyrope_gpu_init(local))
    w = workload(args.workload, args.scale)
    line = bench_workload(args, torch, pg, dist, w, args.steps, args.warmup, rank, world, local)
    sec = None
    if args.secondary == "auto":
        args.secondary = "c4" if args.workload == "c5" else "none"
    if args.secondary and args.secondary != "none" and args.secondary != args.workload:
        # BASELINE config 4 beside the headline config
        w2 = workload(args.secondary, args.secondary_scale if args.secondary_scale > 0 else args.scale)
        try:
            sec = bench_workload(args, torch, pg, dist, w2, args.steps, args.warmup, rank, world, local)
        except Exception as ex:
            if world > 1:
                raise
            sec = {"config": config_of(w2), "error": str(ex)[:300]}
    bad = []
    if rank == 0:
        if sec is not None:
            line["secondary"] = sec
        for blk in (line, sec):
            if blk and blk.get("parity") and blk["parity"].get("mismatch"):
                bad.append(blk["config"]["workload"])
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if bad:
        log(f"PARITY MISMATCH against the oracle in: {bad}")
        sys.exit(3)



def run_sharded_entry(args):
    """bench.py --sharded-entry --gpus N: ONE process drives N GPUs through the library's multi-device entry point
    (pyrope_sharded_*, csrc/sharded.cu) — what a C# GpuVectorIndex P/Invokes.  Same workload, same parity check; `value` is
    batches through pyrope_sharded_search_batch_device (queries and results resident on the first device), `e2e` through
    pyrope_sharded_search_batch (host buffers).  The call is synchronous, so both are wall-clock rates over K calls."""
    import torch

    import pyrope_b200 as pg
    from pyrope_b200 import _lib
    N = args.gpus
    w = workload(args.workload, args.scale)
    assert w["kind"] == "IVF_PQ", "the sharded-entry bench covers the IVF_PQ headline workload"
    nq, dim, k, nprobe = w["nq"], w["dim"], w["topk"], w["nprobe"]
    _lib.check(pg.load().pyrope_gpu_init(0))
    sx = pg.ShardedIndex(N, pg.IVF_PQ, dim, pg.L2, nlist=w["nlist"], m=w["m"], k=w["k"])
    ntrain = min(w["n"], max(40 * w["nlist"], 65536))
    sx.set_train_params(ntrain, 4 if w["nlist"] > 1024 else 10)
    tb0 = time.time()
    chunk = min(w["n"], (1 << 31) // (dim * 4) // 2)
    for r in range(N):  # device-resident feed: every shard sees every row (the lists it does not own are dropped at build)
        shard, dev = sx.shard(r)
        torch.cuda.set_device(dev)
        _lib.check(pg.load().pyrope_gpu_init(dev))
        shard.reserve(w["n"])
        stage = torch.empty(chunk * dim, dtype=torch.float32, device=f"cuda:{dev}")
        row = 0
        while row < w["n"]:
            c = min(chunk, w["n"] - row)
            _lib.fill_uniform_device(stage.data_ptr(), c * dim, 42, row * dim, stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            shard.add_device(stage.data_ptr(), c)
            row += c
        del stage
        torch.cuda.empty_cache()
    sx.note_rows(w["n"])
    tb1 = time.time()
    sx.build()
    tb2 = time.time()
    log(f"sharded entry: {N} shards fed in {tb1 - tb0:.1f}s, built in {tb2 - tb1:.1f}s, {sx.stats()} rows")
    torch.cuda.set_device(0)
    _lib.check(pg.load().pyrope_gpu_init(0))
    Q = make_queries(torch, w)
    sc = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    rw = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    cn = torch.empty((nq,), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    for _ in range(args.warmup):
        sx.search_device(Q.data_ptr(), nq, k, sc.data_ptr(), rw.data_ptr(), cn.data_ptr(), nprobe=nprobe)
    sampler = ClockSampler(0)
    sampler.start()
    dev_ms = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sx.search_device(Q.data_ptr(), nq, k, sc.data_ptr(), rw.data_ptr(), cn.data_ptr(), nprobe=nprobe)
        dev_ms += sx.last_search_ms()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    dump_outputs(args.dump_outputs, w["name"], sc.cpu().numpy(), rw.cpu().numpy(), cn.cpu().numpy())
    Qh = Q.cpu().numpy()
    for _ in range(2):
        hs, hr, hc = sx.search(Qh, k, nprobe=nprobe)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        hs, hr, hc = sx.search(Qh, k, nprobe=nprobe)
    dte = time.perf_counter() - t0
    same = bool(np.array_equal(hr, rw.cpu().numpy()) and np.array_equal(hs, sc.cpu().numpy()))
    cpu, parity = None, None
    if not args.no_cpu:
        oix, _ = build_gpu_index(pg, torch, w, 0, 1)
        oidx, held, note = oracle_index_from_gpu(oix, w, torch)
        oix.close()
        cpu, s, ores = time_cpu_baseline(oidx, held, note, Qh, w, args.cpu_budget)
        parity = compare_topk(ores, (hr[:s], hs[:s], hc[:s]),
                              f"oracle/oracle.c on the unsharded index: merged top-k of {N} GPUs behind pyrope_sharded_search_batch")
        parity["e2e_result_identical_to_device_result"] = same
    line = {"metric": METRIC_NAME, "value": round(nq * args.steps / dt, 1), "unit": "QPS", "n_gpus": N, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 4), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": dtype_of(w), "data": "synthetic uniform[0,1) fp32, counter-based generator",
            "config": config_of(w),
            "details": {"entry": "pyrope_sharded_search_batch_device: one process, one host thread and one stream per device, probe "
                        "lists exchanged by peer stores over NVLink, in-kernel threshold exchange, merge on the first device",
                        "device_ms_per_step_first_device": round(dev_ms / args.steps, 4), "add_s": round(tb1 - tb0, 2),
                        "build_s": round(tb2 - tb1, 2)},
            "clocks": clocks,
            "e2e": {"value": round(nq * args.steps / dte, 1), "unit": "QPS", "h2d_bytes_per_step": nq * dim * 4 * N,
                    "d2h_bytes_per_step": nq * k * 12 + nq * 4},
            "cpu_baseline": cpu, "parity": parity}
    emit(line)
    sx.close()
    if parity and parity.get("mismatch"):
        sys.exit(3)


def run_reference(args):
    """The reference's own CPU implementation of the path.  The C# engine cannot be built in this image
    (no dotnet), so this arm times the oracle port of its loops (oracle/oracle.c) with all host threads,
    on the same config; the index it searches is the one the GPU builds (setup only, untimed)."""
    rank, world, local = dist_env()
    if rank != 0:
        return
    import torch

    import pyrope_b200 as pg
    from pyrope_b200 import _lib
    torch.cuda.set_device(0)
    _lib.check(pg.load().pyrope_gpu_init(0))
    w = workload(args.workload, args.scale)
    ix, build_info = build_gpu_index(pg, torch, w, 0, 1)
    Q = make_queries(torch, w)
    Qh = Q.cpu().numpy()
    oidx, held, note = oracle_index_from_gpu(ix, w, torch)
    del ix
    torch.cuda.empty_cache()
    threads = host_cores()
    # size one step to ~ (budget / (steps+warmup)) seconds
    probe = min(len(Qh), 2 * threads)
    t0 = time.perf_counter()
    _osearch(oidx, Qh[:probe], w, threads)
    per_q = (time.perf_counter() - t0) / probe
    per_step_budget = max(1.0, args.cpu_budget * 6 / max(1, args.steps + args.warmup))
    s = int(max(threads, min(len(Qh), per_step_budget / max(per_q, 1e-9))))
    for i in range(args.warmup):
        _osearch(oidx, Qh[:s], w, threads)
    t0 = time.perf_counter()
    for i in range(args.steps):
        off = (i * s) % max(1, len(Qh) - s + 1)
        ids, scores, counts = _osearch(oidx, Qh[off:off + s], w, threads)
    dt = time.perf_counter() - t0
    dump_outputs(args.dump_outputs, w["name"], scores, ids, counts)
    value = s * args.steps / dt * (held / w["n"])
    sample = f"{s} of the batch's {len(Qh)} queries per step over {note}, one query per thread"
    line = {"impl": "reference", "metric": METRIC_NAME, "value": round(value, 2), "unit": "QPS", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dtype_of(w),
            "data": "synthetic uniform[0,1) fp32 (same generator and seeds as the GPU arm)",
            "config": config_of(w), "details": {**build_info, "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")},
            "cpu_baseline": {"value": round(value, 2), "unit": "QPS", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": round(value, 2), "unit": "QPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line goes to the real stdout; everything libraries print (NCCL's version banner, ...) was
    redirected to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # fd 1 -> stderr for the rest of the process (native libraries included)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("PYROPE_BENCH_WORKLOAD", "c5"))
    ap.add_argument("--scale", type=float, default=float(os.environ.get("PYROPE_BENCH_SCALE", "1.0")))
    ap.add_argument("--secondary", default=os.environ.get("PYROPE_BENCH_SECONDARY", "auto"),
                    help="workload reported as the line's `secondary` block (auto = c4 beside c5, none = skip)")
    ap.add_argument("--secondary-scale", type=float, default=float(os.environ.get("PYROPE_BENCH_SECONDARY_SCALE", "0")))
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU-baseline work")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline AND the parity check against the oracle")
    ap.add_argument("--no-threshold-exchange", action="store_true",
                    help="multi-GPU IVF_PQ: do not share thresholds between the ranks' scan kernels")
    ap.add_argument("--nccl-exchange", action="store_true",
                    help="multi-GPU: all-gather probe lists and results with NCCL instead of the library's peer-memory exchange")
    ap.add_argument("--recall-queries", type=int, default=200, help="queries used for the recall@10 read-out (0 = skip)")
    ap.add_argument("--sharded-entry", action="store_true",
                    help="one process drives --gpus N devices through pyrope_sharded_* (no torchrun)")
    ap.add_argument("--profile-step", action="store_true",
                    help="bracket one extra search step with cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--flat-parity-queries", type=int, default=32,
                    help="queries of a full-size FLAT batch checked against the independent exact top-k")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step as DIR/<workload>_{scores,ids,counts}.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        run_reference(args)
    elif args.sharded_entry:
        run_sharded_entry(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
