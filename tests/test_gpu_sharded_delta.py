"""The multi-GPU index as a server holds it: the row-ordinal surface of pyrope_sharded_* that IVectorIndex needs beyond
add / delete / build / search (Upsert, shadowing, labels, centroids, codebooks, Snapshot / Load), Head+Tail with a
sharded tail (pyrope_delta_create_sharded) and string ids over N GPUs (pyrope_vindex_create_sharded).  Every result must
equal the single-device index's: identical ids, bit-identical scores.  Runs for each device count the box has."""
import ctypes as C
import os
import shutil
import struct

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.test_gpu_vector_index import RefDelta, _check

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    import pyrope_b200 as pg
    pg._lib.check(pg.load().pyrope_gpu_init(0))
    return pg


@pytest.fixture(scope="module")
def vi(gpu):
    from pyrope_b200 import vector_index
    return vector_index


def _ndev(gpu):
    n = C.c_int32(0)
    gpu._lib.check(gpu.load().pyrope_gpu_device_count(C.byref(n)))
    return n.value


def _counts(gpu):
    return [c for c in (1, 2, 4, 8) if c <= _ndev(gpu)]


def _same(a, b, ctx):
    """(scores, rows, counts) of two searches: identical counts and ids, bit-identical scores."""
    np.testing.assert_array_equal(a[2], b[2], err_msg=f"{ctx}: counts")
    for q in range(len(a[2])):
        c = int(a[2][q])
        np.testing.assert_array_equal(a[1][q][:c], b[1][q][:c], err_msg=f"{ctx} q{q}: ids")
        np.testing.assert_array_equal(a[0][q][:c], b[0][q][:c], err_msg=f"{ctx} q{q}: scores")


def _same_results(a, b, ctx):
    """two SearchBatch results of the string-id classes"""
    assert len(a) == len(b)
    for q, (x, y) in enumerate(zip(a, b)):
        assert [r.Id for r in x] == [r.Id for r in y], f"{ctx} q{q}: ids"
        assert [r.Score for r in x] == [r.Score for r in y], f"{ctx} q{q}: scores"


KINDS = {"FLAT": 0, "IVF_FLAT": 1, "IVF_PQ": 2}
DIM, NLIST, M, K = 32, 16, 8, 64


def _make(gpu, kind, n):
    one = gpu.GpuIndex(KINDS[kind], DIM, gpu.L2, nlist=NLIST, m=M, k=K)
    sx = gpu.ShardedIndex(n, KINDS[kind], DIM, gpu.L2, nlist=NLIST, m=M, k=K)
    return one, sx


def _populate(gpu, kind, ix):
    """add / build / add / update / shadow / delete, the same on a GpuIndex and a ShardedIndex"""
    rng = np.random.default_rng(5)
    X = rng.random((5000, DIM), dtype=np.float32)
    ix.add(X[:4000], labels=np.arange(4000) + 100_000)
    ix.build()
    ix.add(X[4000:4600], labels=np.arange(4000, 4600) + 100_000)
    ix.update_row(4100, X[4700])                                                  # a buffered (FLAT: any) row, in place
    assert ix.delete_row(4200)
    if kind == "FLAT":
        assert ix.delete_row(5)
        ix.update_row(5, X[4800])                                                 # Upsert un-deletes
    else:
        with pytest.raises(gpu.PyropeGpuError) as e:
            ix.update_row(10, X[4900])                                            # a list row
        assert e.value.code == gpu._lib.ERR_NOT_FOUND
        ix.shadow_row(11)
        ix.shadow_row(12)
        ix.shadow_row(12, False)
    return rng.random((64, DIM), dtype=np.float32)


def _stats(ix):
    s = ix.stats()
    return s["live"] if isinstance(s, dict) else s


@pytest.mark.parametrize("kind", list(KINDS))
def test_row_ordinal_surface_matches_single_device(gpu, kind):
    for n in _counts(gpu):
        one, sx = _make(gpu, kind, n)
        Q = _populate(gpu, kind, one)
        _populate(gpu, kind, sx)
        assert _stats(one) == sx.stats()
        for k, nprobe in ((10, 4), (1, 16), (50, 8)):
            _same(one.search(Q, k, nprobe=nprobe), sx.search(Q, k, nprobe=nprobe), f"{kind} n={n} k={k}")
        if kind != "FLAT":
            assert sx.is_built()
            assert one.centroids().tobytes() == sx.centroids().tobytes()
        if kind == "IVF_PQ":
            a, b = one.codebooks(), sx.codebooks()
            assert a[0].tobytes() == b[0].tobytes() and np.array_equal(a[1], b[1])
        # labels: every row relabelled, both sides alike
        lab = np.arange(4600, dtype=np.int64)[::-1].copy()
        gpu._lib.check(gpu.load().pyrope_index_set_labels(one._h, lab.size, gpu._lib._p(lab)))
        sx.set_labels(lab)
        _same(one.search(Q, 10, nprobe=4), sx.search(Q, 10, nprobe=4), f"{kind} n={n} relabelled")
        sx.close()


def _manifest(path):
    """(shard count, [(shard file name, offset of its recorded byte count)]) of a sharded snapshot manifest"""
    b = open(path, "rb").read()
    assert b[:8] == b"PYRSHD01"
    n = struct.unpack_from("<i", b, 12)[0]
    nsegs = struct.unpack_from("<q", b, 56)[0]
    o = 64 + 28 * nsegs + 8 * n
    out = []
    for _ in range(n):
        ln = struct.unpack_from("<I", b, o)[0]
        out.append((b[o + 4:o + 4 + ln].decode(), o + 4 + ln))
        o += 4 + ln + 8
    return n, out


@pytest.mark.parametrize("kind", list(KINDS))
def test_snapshot_round_trip(gpu, kind, tmp_path):
    for n in _counts(gpu):
        _, sx = _make(gpu, kind, n)
        Q = _populate(gpu, kind, sx)
        want = [sx.search(Q, k, nprobe=p) for k, p in ((10, 4), (50, 16))]
        path = str(tmp_path / f"{kind}_{n}.snap")
        sx.snapshot(path)
        _, files1 = _manifest(path)
        assert all(os.path.exists(str(tmp_path / f)) and ".g1.shard" in f for f, _ in files1)
        _, ld = _make(gpu, kind, n)
        ld.load(path)
        assert ld.stats() == sx.stats()
        for (k, p), w in zip(((10, 4), (50, 16)), want):
            for rep in range(2):                                                   # repeated batches after a load
                _same(w, ld.search(Q, k, nprobe=p), f"{kind} n={n} loaded k={k} rep={rep}")
        if kind != "FLAT":
            assert ld.centroids().tobytes() == sx.centroids().tobytes()
        # a second snapshot to the same path: the first generation's shard files go once the manifest names the second
        sx.snapshot(path)
        _, files2 = _manifest(path)
        assert all(".g2.shard" in f and os.path.exists(str(tmp_path / f)) for f, _ in files2)
        assert not any(os.path.exists(str(tmp_path / f)) for f, _ in files1)
        sx.close()
        ld.close()


def _copy_set(src, dst_dir):
    os.makedirs(dst_dir, exist_ok=True)
    _, files = _manifest(src)
    shutil.copy(src, os.path.join(dst_dir, "m.snap"))
    for f, _ in files:
        shutil.copy(os.path.join(os.path.dirname(src), f), os.path.join(dst_dir, f))
    return os.path.join(dst_dir, "m.snap")


@pytest.mark.parametrize("kind", ["FLAT", "IVF_PQ"])
def test_failed_load_leaves_the_index_untouched(gpu, kind, tmp_path):
    E = gpu._lib
    for n in _counts(gpu):
        _, a = _make(gpu, kind, n)
        Q = _populate(gpu, kind, a)
        pa = str(tmp_path / f"a{n}.snap")
        a.snapshot(pa)
        _, b = _make(gpu, kind, n)                                                 # another snapshot, other rows
        b.add(np.random.default_rng(9).random((3000, DIM), dtype=np.float32))
        b.build()
        pb = str(tmp_path / f"b{n}.snap")
        b.snapshot(pb)
        single = gpu.GpuIndex(KINDS[kind], DIM, gpu.L2, nlist=NLIST, m=M, k=K)
        single.add(np.ones((4, DIM), np.float32))
        ps = str(tmp_path / f"single{n}.snap")
        single.snapshot(ps)
        _, t = _make(gpu, kind, n)
        _populate(gpu, kind, t)
        t.add(np.full((3, DIM), 0.5, np.float32))                                  # t differs from both snapshots
        before = t.search(Q, 10, nprobe=4)
        stats_before = t.stats()

        def fails(path, code, ctx, *words):
            with pytest.raises(gpu.PyropeGpuError) as e:
                t.load(path)
            assert e.value.code == code, f"{ctx}: {e.value}"
            for w in words:
                assert w in e.value.message, f"{ctx}: {e.value.message}"
            _same(before, t.search(Q, 10, nprobe=4), f"{kind} n={n} after failed load ({ctx})")
            assert t.stats() == stats_before

        # wrong device count
        p = _copy_set(pa, str(tmp_path / f"count{n}"))
        raw = bytearray(open(p, "rb").read())
        struct.pack_into("<i", raw, 12, n + 1 if n < 8 else n - 1)
        open(p, "wb").write(bytes(raw))
        fails(p, E.ERR_INVALID_ARG, "device count", str(n), str(n + 1 if n < 8 else n - 1))
        # a single-device snapshot
        fails(ps, E.ERR_INVALID_ARG, "single-device snapshot", "single-device")
        # one shard file truncated: caught by the recorded size, and by the shard's own parse when the size is patched
        p = _copy_set(pa, str(tmp_path / f"trunc{n}"))
        _, files = _manifest(p)
        f, off = files[-1]
        fp = os.path.join(os.path.dirname(p), f)
        size = os.path.getsize(fp)
        with open(fp, "r+b") as fh:
            fh.truncate(size // 2)
        fails(p, E.ERR_INVALID_ARG, "truncated shard file")
        raw = bytearray(open(p, "rb").read())
        struct.pack_into("<Q", raw, off, size // 2)
        open(p, "wb").write(bytes(raw))
        fails(p, E.ERR_INVALID_ARG, "truncated shard file, size patched")
        # a shard file missing
        p = _copy_set(pa, str(tmp_path / f"missing{n}"))
        os.remove(os.path.join(os.path.dirname(p), _manifest(p)[1][0][0]))
        fails(p, E.ERR_NOT_FOUND, "missing shard file")
        # a shard file swapped in from another snapshot (size patched too, so the shard's row count is what differs)
        p = _copy_set(pa, str(tmp_path / f"swap{n}"))
        _, files = _manifest(p)
        f, off = files[-1]
        other = os.path.join(os.path.dirname(pb), _manifest(pb)[1][-1][0])
        shutil.copy(other, os.path.join(os.path.dirname(p), f))
        fails(p, E.ERR_INVALID_ARG, "swapped shard file, recorded size")
        raw = bytearray(open(p, "rb").read())
        struct.pack_into("<Q", raw, off, os.path.getsize(other))
        open(p, "wb").write(bytes(raw))
        fails(p, E.ERR_INVALID_ARG, "swapped shard file", "manifest expects")
        # and the intact set still loads
        t.load(pa)
        _same(a.search(Q, 10, nprobe=4), t.search(Q, 10, nprobe=4), f"{kind} n={n} good load")
        for ix in (a, b, t):
            ix.close()


# ------------------------------------------------------------------ Head+Tail with a sharded tail
@pytest.mark.parametrize("tail_kind", ["IVF_FLAT", "IVF_PQ"])
def test_sharded_delta_random_sequence(gpu, vi, tail_kind):
    """test_delta_random_sequence_matches_oracle's op sequence on create_index(..., {"devices": n}) against the
    single-device create_index, and against the oracle's RefDelta for the largest n."""
    dim, n0 = 16, 1500
    rng = np.random.default_rng(11)
    base = rng.random((n0 + 600, dim), dtype=np.float32)
    Q = rng.random((24, dim), dtype=np.float32)
    params = {"nlist": 12, "m": 4, "k": 64}
    counts = _counts(gpu)
    for n in counts:
        one = vi.create_index(tail_kind, dim, vi.VectorMetric.L2, params)
        shd = vi.create_index(tail_kind, dim, vi.VectorMetric.L2, dict(params, devices=n))
        ref = None
        if n == counts[-1]:
            rt = orc.IvfFlatIndex(dim, orc.L2, nlist=12) if tail_kind == "IVF_FLAT" else orc.IvfPqIndex(dim, orc.L2, m=4, k=64, nlist=12)
            ref = RefDelta(dim, orc.L2, rt)

        def both(fn):
            a, b = fn(one), fn(shd)
            assert a == b
            return a

        def check(ctx, ks=(10,), **kw):
            opts = vi.SearchOptions(MaxScans=kw.get("max_scans"), NProbe=kw.get("nprobe"))
            for k in ks:
                _same_results(one.SearchBatch(Q, k, opts), shd.SearchBatch(Q, k, opts), f"{tail_kind} n={n} {ctx} k={k}")
                if ref is not None:
                    _check(ref, shd, vi, Q, k, f"{tail_kind} n={n} {ctx} k={k} vs oracle", **kw)
            assert one.GetStats() == shd.GetStats()

        for i in range(n0):
            for ix in (one, shd):
                ix.Upsert(f"v{i}", base[i])
            if ref:
                ref.add(i, base[i])
        check("head only")
        for ix in (one, shd):
            ix.Build()
        if ref:
            ref.build()
        assert np.array_equal(np.stack(one.GetCentroids()), np.stack(shd.GetCentroids()))
        check("after first compaction", nprobe=4)
        for i in range(n0, n0 + 300):
            for ix in (one, shd):
                ix.Upsert(f"v{i}", base[i])
            if ref:
                ref.add(i, base[i])
        for j, i in enumerate(range(0, n0, 25)):                                   # overwrites of ids that live in the tail
            v = base[n0 + 300 + j]
            for ix in (one, shd):
                ix.Upsert(f"v{i}", v)
            if ref:
                ref.add(i, v)
        dels = list(range(n0 + 5, n0 + 300, 30))
        if tail_kind == "IVF_FLAT":
            dels += list(range(3, n0, 40))
        for i in dels:
            r = both(lambda ix: ix.Delete(f"v{i}"))
            if ref:
                assert ref.delete(i) == r
        check("head over tail", ks=(1, 10, 50), nprobe=4)
        check("head over tail, all lists", ks=(10,), nprobe=12)
        for ix in (one, shd):
            ix.Build()
        if ref:
            ref.build()
        assert np.array_equal(np.stack(one.GetCentroids()), np.stack(shd.GetCentroids()))
        check("after second compaction", ks=(1, 10, 50), nprobe=4)
        assert shd._head.GetStats().Count == 0


def test_sharded_delta_head_id_in_tail_top_k(gpu, vi):
    """The head holds an id from the tail's top k: the tail still contributes only k - 1 entries (the reference asks
    the tail for topK and de-duplicates afterwards), not its (k+1)-th."""
    dim = 8
    rng = np.random.default_rng(4)
    X = rng.random((40, dim), dtype=np.float32)
    q = X[0] + 0.01
    for n in _counts(gpu):
        d = vi.create_index("IVF_FLAT", dim, vi.VectorMetric.L2, {"nlist": 2, "devices": n})
        one = vi.create_index("IVF_FLAT", dim, vi.VectorMetric.L2, {"nlist": 2})
        for ix in (d, one):
            for i in range(40):
                ix.Add(f"v{i}", X[i])
            ix.Build()
        opts = vi.SearchOptions(NProbe=2)
        tail4 = d.Search(q, 4, opts)
        far = np.full(dim, 50.0, np.float32)
        for ix in (d, one):
            ix.Upsert(tail4[1].Id, far)                                            # the head now holds the tail's 2nd id
        got = d.Search(q, 3, opts)
        assert [r.Id for r in got] == [tail4[0].Id, tail4[2].Id, tail4[1].Id], f"n={n}"
        assert got[2].Score < tail4[3].Score                                       # the head's copy ranks last
        assert tail4[3].Id not in [r.Id for r in got]
        _same_results([got], [one.Search(q, 3, opts)], f"n={n} head id in tail top k")


def test_sharded_delta_max_scans(gpu, vi):
    dim = 16
    rng = np.random.default_rng(2)
    X = rng.random((800, dim), dtype=np.float32)
    Q = rng.random((8, dim), dtype=np.float32)
    opts = vi.SearchOptions(MaxScans=60, NProbe=4)
    for n in _counts(gpu):
        for kind in ("IVF_PQ", "IVF_FLAT"):
            params = {"nlist": 8, "m": 4, "k": 32}
            one = vi.create_index(kind, dim, vi.VectorMetric.L2, params)
            shd = vi.create_index(kind, dim, vi.VectorMetric.L2, dict(params, devices=n))
            for ix in (one, shd):
                for i in range(600):
                    ix.Add(f"v{i}", X[i])
                ix.Build()
                for i in range(600, 800):
                    ix.Add(f"v{i}", X[i])
            if kind == "IVF_FLAT" and n > 1:                                       # the budget cannot be split over devices
                with pytest.raises(gpu.PyropeGpuError) as e:
                    shd.SearchBatch(Q, 10, opts)
                assert e.value.code == gpu._lib.ERR_UNSUPPORTED
            else:
                _same_results(one.SearchBatch(Q, 10, opts), shd.SearchBatch(Q, 10, opts), f"{kind} n={n} MaxScans")


def test_sharded_string_ids_snapshot_load(gpu, vi, tmp_path):
    dim = 8
    rng = np.random.default_rng(3)
    X = rng.random((300, dim), dtype=np.float32)
    opts = vi.SearchOptions(NProbe=4)
    for n in _counts(gpu):
        made = [vi.create_index("IVF_FLAT", dim, vi.VectorMetric.L2, {"nlist": 4, "devices": n}),
                vi.IvfPqVectorIndex(dim, vi.VectorMetric.L2, m=4, k=32, nList=4, devices=n)]
        for j, d in enumerate(made):
            for i in range(250):
                d.Add(f"v{i}", X[i])
            d.Build()
            for i in range(250, 300):
                d.Add(f"v{i}", X[i])
            d.Upsert("v270", X[270] * 0.25)
            path = str(tmp_path / f"s{n}_{j}.snap")
            d.Snapshot(path)
            e = (vi.create_index("IVF_FLAT", dim, vi.VectorMetric.L2, {"nlist": 4, "devices": n}) if j == 0
                 else vi.IvfPqVectorIndex(dim, vi.VectorMetric.L2, m=4, k=32, nList=4, devices=n))
            e.Load(path)
            _same_results(d.SearchBatch(X[::37], 5, opts), e.SearchBatch(X[::37], 5, opts), f"n={n} {j} loaded")
            assert e.GetStats() == d.GetStats()
            assert e.Delete("v270") and not e.Delete("v270")
            assert "v270" not in [r.Id for r in e.Search(X[270] * 0.25, 5, opts)]
            if j == 1:
                with pytest.raises(vi.InvalidOperationException):
                    e.native()


def test_sharded_delta_construction_errors(gpu, vi):
    L = gpu.load()
    E = gpu._lib
    n = _counts(gpu)[-1]
    # a FLAT tail cannot be sharded under a Head+Tail
    head = gpu.GpuIndex(gpu.FLAT, 16, gpu.L2, device=0)
    flat = gpu.ShardedIndex(n, gpu.FLAT, 16, gpu.L2)
    d = E.vp()
    assert L.pyrope_delta_create_sharded(head._h, flat._s, C.byref(d)) == E.ERR_UNSUPPORTED
    with pytest.raises(gpu.PyropeGpuError):
        vi.create_index("FLAT", 16, vi.VectorMetric.L2, {"devices": n})
    # dimension / metric as pyrope_delta_create
    ivf = gpu.ShardedIndex(n, gpu.IVF_FLAT, 16, gpu.L2, nlist=4)
    other = gpu.GpuIndex(gpu.FLAT, 8, gpu.L2, device=0)
    assert L.pyrope_delta_create_sharded(other._h, ivf._s, C.byref(d)) == E.ERR_INVALID_ARG
    assert L.pyrope_delta_create_sharded(head._h, ivf._s, C.byref(d)) == E.OK
    assert L.pyrope_delta_destroy(d) == E.OK
    if _ndev(gpu) >= 2:                                                            # the head must live on the tail's first device
        away = gpu.GpuIndex(gpu.FLAT, 16, gpu.L2, device=1)
        assert L.pyrope_delta_create_sharded(away._h, ivf._s, C.byref(d)) == E.ERR_INVALID_ARG
        assert b"device" in L.pyrope_last_error()
        away.close()
        gpu._lib.check(L.pyrope_gpu_init(0))
    for ix in (head, flat, ivf, other):
        ix.close()
