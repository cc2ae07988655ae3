"""Extend: the write buffer of a built IVF index joins its inverted lists without re-training (pyrope_index_extend,
pyrope_sharded_extend, pyrope_delta_extend_tail, pyrope_vindex_extend).  The lists must equal, bit for bit, the old lists
plus each buffered row appended to its nearest current centroid's list (add order), IVF_PQ rows encoded with the current
codebooks; searches must match the CPU oracle over those lists; a sharded Extend must equal the one-device one."""
import ctypes as C
import threading

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.parity import assert_batch_equivalent, assert_topk_equivalent

DIM, K = 32, 64


@pytest.fixture(scope="module")
def gpu():
    import pyrope_b200 as pg
    pg._lib.check(pg.load().pyrope_gpu_init(0))
    return pg


@pytest.fixture(scope="module")
def vi(gpu):
    from pyrope_b200 import vector_index
    return vector_index


def _counts(gpu):
    n = C.c_int32(0)
    gpu._lib.check(gpu.load().pyrope_gpu_device_count(C.byref(n)))
    return [c for c in (1, 2, 4, 8) if c <= n.value]


def _same(a, b, ctx):
    """(scores, rows, counts) of two searches: identical counts and ids, bit-identical scores."""
    np.testing.assert_array_equal(a[2], b[2], err_msg=f"{ctx}: counts")
    for q in range(len(a[2])):
        c = int(a[2][q])
        np.testing.assert_array_equal(a[1][q][:c], b[1][q][:c], err_msg=f"{ctx} q{q}: ids")
        np.testing.assert_array_equal(a[0][q][:c], b[0][q][:c], err_msg=f"{ctx} q{q}: scores")


def _expected(off, rows, codes, new_rows, Xall, cent, metric, pq=None):
    """old lists + every new row (add order) appended to its nearest centroid's list -> (off, rows, codes)"""
    nc = len(off) - 1
    lists = [list(rows[off[c]:off[c + 1]]) for c in range(nc)]
    lcodes = [list(codes[off[c]:off[c + 1]]) for c in range(nc)] if pq is not None else None
    for r in new_rows:
        a = orc.find_nearest_centroid(Xall[r], cent, metric)
        lists[a].append(r)
        if pq is not None:
            lcodes[a].append(pq.encode((Xall[r] - cent[a]).astype(np.float32)))
    eoff = np.zeros(nc + 1, np.int64)
    eoff[1:] = np.cumsum([len(x) for x in lists])
    erows = np.array([r for x in lists for r in x], np.int64)
    ecodes = np.array([c for x in lcodes for c in x], np.uint8).reshape(-1, pq.m) if pq is not None else None
    return eoff, erows, ecodes


def _oracle_pq(g):
    cb, ks = g.codebooks()
    pq = orc.ProductQuantizer(DIM, g.m, g.k)
    pq.set_codebook(cb, ks)
    return pq, cb


CASES = [  # (kind, metric, m, nlist, n0, n1)
    ("ivf_flat", orc.L2, 0, 24, 3000, 700),
    ("ivf_flat", orc.IP, 0, 24, 3000, 700),
    ("ivf_flat", orc.COSINE, 0, 24, 3000, 700),
    ("ivf_pq", orc.L2, 4, 24, 3000, 700),
    ("ivf_pq", orc.L2, 8, 24, 3000, 700),
    ("ivf_pq", orc.L2, 16, 24, 3000, 700),
    ("ivf_flat", orc.L2, 0, 2048, 6000, 1500),  # assignment through the tensor-core shortlist
]


def _new(gpu, kind, metric, m, nlist):
    return gpu.GpuIndex(gpu.IVF_PQ if kind == "ivf_pq" else gpu.IVF_FLAT, DIM, metric, nlist=nlist, m=max(m, 4), k=K)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[f"{c[0]}-metric{c[1]}-m{c[2]}-nlist{c[3]}" for c in CASES])
def test_extend_lists_bit_exact_and_search(gpu, case):
    kind, metric, m, nlist, n0, n1 = case
    rng = np.random.default_rng(7 + nlist + m + metric)
    X = rng.standard_normal((n0 + n1, DIM)).astype(np.float32)
    Q = rng.standard_normal((48, DIM)).astype(np.float32)
    g = _new(gpu, kind, metric, m, nlist)
    if nlist >= 2048:
        g.set_train_params(0, 2)
    g.add(X[:n0])
    g.build()
    off0, rows0, codes0 = g.lists()
    assert g.add(X[n0:]) == n0
    g.extend()
    assert g.stats()["buffer"] == 0
    off, rows, codes = g.lists()
    cent = g.centroids()
    pq, cb = _oracle_pq(g) if kind == "ivf_pq" else (None, None)
    eoff, erows, ecodes = _expected(off0, rows0, codes0, range(n0, n0 + n1), X, cent, metric, pq)
    np.testing.assert_array_equal(off, eoff)
    np.testing.assert_array_equal(rows, erows)
    if pq is not None:
        np.testing.assert_array_equal(codes, ecodes)

    # the same lists as a Build with the centroids (and codebooks) frozen, fed old rows then new ones
    f = _new(gpu, kind, metric, m, nlist)
    f.set_codebooks(cent, cb)
    f.add(X)
    f.build()
    foff, frows, fcodes = f.lists()
    np.testing.assert_array_equal(foff, off)
    np.testing.assert_array_equal(frows, rows)
    if pq is not None:
        np.testing.assert_array_equal(fcodes, codes)

    # search over the extended lists against the oracle holding the expected lists
    if kind == "ivf_pq":
        ref = orc.IvfPqIndex(DIM, metric, m=m, k=K, nlist=nlist)
        ref.adopt(cent, cb, eoff, erows, ecodes)
    else:
        ref = orc.IvfFlatIndex(DIM, metric, nlist=nlist)
        ref.adopt(cent, eoff, erows, X[erows])
    for nprobe in (1, 3, 8):
        for k in (10, 100):
            budgets = (-1, 50, 700) if kind == "ivf_flat" else (-1,)
            for ms in budgets:
                want = ref.search_batch(Q, k, max_scans=ms, nprobe=nprobe)
                sc, rw, cn = g.search(Q, k, max_scans=ms, nprobe=nprobe)
                assert_batch_equivalent(want, (rw, sc, cn), ctx=f"{case} nprobe={nprobe} k={k} ms={ms}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["ivf_flat", "ivf_pq"])
def test_extend_dead_and_shadowed_entries(gpu, kind):
    m, nlist, n0 = 8, 16, 2500
    rng = np.random.default_rng(21)
    X = rng.standard_normal((n0 + 900, DIM)).astype(np.float32)
    Q = rng.standard_normal((32, DIM)).astype(np.float32)
    g = _new(gpu, kind, orc.L2, m, nlist)
    label = {}
    g.add(X[:n0], labels=np.arange(n0))
    for r in range(n0):
        label[r] = r
    g.build()
    off0, rows0, codes0 = g.lists()
    dead = set()
    if kind == "ivf_flat":  # IVF_PQ deletes only buffered rows
        for r in range(0, n0, 37):
            assert g.delete_row(r)
            dead.add(r)
    # Upsert of indexed ids: a buffered copy under the same label shadows the list entry
    upserted = [r for r in range(5, n0, 53) if r not in dead]
    for i, r in enumerate(upserted):
        nr = g.add(X[n0 + i], labels=[r])
        label[nr] = r
        g.shadow_row(r)
        dead.add(r)
    nxt = n0 + len(upserted)
    fresh = g.add(X[nxt:n0 + 900], labels=np.arange(nxt, n0 + 900) + 100_000)
    for r in range(fresh, fresh + (n0 + 900 - nxt)):
        label[r] = r - fresh + nxt + 100_000
    Xrow = {r: X[r] for r in range(n0)}
    Xrow.update({n0 + i: X[n0 + i] for i in range(len(upserted))})
    Xrow.update({r: X[r - fresh + nxt] for r in range(fresh, fresh + (n0 + 900 - nxt))})
    g.extend()
    # shadowed entries are now deleted: no longer addressable, not even to un-shadow them
    for r in upserted:
        with pytest.raises(gpu.PyropeGpuError) as e:
            g.shadow_row(r, False)
        assert e.value.code == gpu._lib.ERR_NOT_FOUND
    off, rows, codes = g.lists()
    cent = g.centroids()
    pq, cb = _oracle_pq(g) if kind == "ivf_pq" else (None, None)
    Xall = np.zeros((max(Xrow) + 1, DIM), np.float32)
    for r, v in Xrow.items():
        Xall[r] = v
    new_rows = list(range(n0, n0 + len(upserted))) + list(range(fresh, fresh + (n0 + 900 - nxt)))
    eoff, erows, ecodes = _expected(off0, rows0, codes0, new_rows, Xall, cent, orc.L2, pq)
    np.testing.assert_array_equal(off, eoff)
    np.testing.assert_array_equal(rows, erows)
    if pq is not None:
        np.testing.assert_array_equal(codes, ecodes)
    # the oracle holds the live entries only, in list order (a MaxScans budget never counts a dead entry)
    keep = np.array([r not in dead for r in erows], bool)
    loff = np.zeros(len(eoff), np.int64)
    for c in range(len(eoff) - 1):
        loff[c + 1] = loff[c] + keep[eoff[c]:eoff[c + 1]].sum()
    lrows = erows[keep]
    if kind == "ivf_pq":
        ref = orc.IvfPqIndex(DIM, orc.L2, m=m, k=K, nlist=nlist)
        ref.adopt(cent, cb, loff, lrows, ecodes[keep])
    else:
        ref = orc.IvfFlatIndex(DIM, orc.L2, nlist=nlist)
        ref.adopt(cent, loff, lrows, Xall[lrows])
    for nprobe in (2, 6):
        for ms in ((-1, 40, 400) if kind == "ivf_flat" else (-1,)):
            want = ref.search_batch(Q, 10, max_scans=ms, nprobe=nprobe)
            wids = np.vectorize(lambda r: label.get(int(r), -1))(want[0]) if want[0].size else want[0]
            sc, rw, cn = g.search(Q, 10, max_scans=ms, nprobe=nprobe)
            assert_batch_equivalent((wids, want[1], want[2]), (rw, sc, cn), ctx=f"{kind} nprobe={nprobe} ms={ms}")
    if kind == "ivf_flat":  # a later Build holds every live id exactly once
        g.build()
        _, brows, _ = g.lists()
        got = sorted(label[int(r)] for r in brows)
        live = sorted(label[r] for r in erows if r not in dead)
        assert got == live


@pytest.mark.gpu
def test_extend_errors(gpu):
    L = gpu.load()
    f = gpu.GpuIndex(gpu.FLAT, DIM, gpu.L2)
    f.add(np.ones((4, DIM), np.float32))
    assert L.pyrope_index_extend(f._h) == gpu._lib.ERR_UNSUPPORTED
    for kind in (gpu.IVF_FLAT, gpu.IVF_PQ):
        g = gpu.GpuIndex(kind, DIM, gpu.L2, nlist=4, m=4, k=16)
        g.add(np.random.default_rng(1).random((64, DIM), dtype=np.float32))
        assert L.pyrope_index_extend(g._h) == gpu._lib.ERR_INVALID_STATE
        assert g.stats()["buffer"] == 64
        g.build()
        off, rows, _ = g.lists()
        g.extend()  # empty buffer: nothing changes
        off2, rows2, _ = g.lists()
        np.testing.assert_array_equal(off, off2)
        np.testing.assert_array_equal(rows, rows2)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["ivf_flat", "ivf_pq"])
def test_extend_sharded_equals_one_device_and_snapshot(gpu, kind, tmp_path):
    nlist, m = 20, 8
    rng = np.random.default_rng(33)
    X = rng.standard_normal((4000, DIM)).astype(np.float32)
    Q = rng.standard_normal((40, DIM)).astype(np.float32)
    code = gpu.IVF_PQ if kind == "ivf_pq" else gpu.IVF_FLAT
    one = gpu.GpuIndex(code, DIM, gpu.L2, nlist=nlist, m=m, k=K)
    one.add(X[:3000])
    one.build()
    one.add(X[3000:3600])
    one.extend()
    one.add(X[3600:])  # a second Extend on top of the first
    one.extend()
    ooff, orows, ocodes = one.lists()
    want = one.search(Q, 20, nprobe=5)
    # one device: snapshot / load round trip
    p = str(tmp_path / f"one_{kind}.bin")
    one.snapshot(p)
    back = gpu.GpuIndex(code, DIM, gpu.L2, nlist=nlist, m=m, k=K)
    back.load(p)
    for a, b in zip(back.lists(), (ooff, orows, ocodes)):
        if b is not None:
            np.testing.assert_array_equal(a, b)
    _same(want, back.search(Q, 20, nprobe=5), f"{kind} one-device reload")
    for n in _counts(gpu):
        sx = gpu.ShardedIndex(n, code, DIM, gpu.L2, nlist=nlist, m=m, k=K)
        sx.add(X[:3000])
        sx.build()
        sx.add(X[3000:3600])
        sx.extend()
        sx.add(X[3600:])
        sx.extend()
        _same(want, sx.search(Q, 20, nprobe=5), f"{kind} n={n}")
        for r in range(n):
            sh, _ = sx.shard(r)
            soff, srows, scodes = sh.lists()
            for c in range(nlist):
                a0, a1 = soff[c], soff[c + 1]
                b0, b1 = ooff[c], ooff[c + 1]
                if c % n == r:
                    np.testing.assert_array_equal(srows[a0:a1], orows[b0:b1], err_msg=f"n={n} shard {r} list {c}")
                    if ocodes is not None:
                        np.testing.assert_array_equal(scodes[a0:a1], ocodes[b0:b1])
                else:
                    assert a1 == a0, f"n={n} shard {r} holds foreign list {c}"
            del sh
        ps = str(tmp_path / f"sharded_{kind}_{n}.bin")
        sx.snapshot(ps)
        sy = gpu.ShardedIndex(n, code, DIM, gpu.L2, nlist=nlist, m=m, k=K)
        sy.load(ps)
        _same(want, sy.search(Q, 20, nprobe=5), f"{kind} n={n} reload")
        sy.close()
        sx.close()


@pytest.mark.gpu
def test_sharded_build_and_extend_are_all_or_nothing(gpu):
    """Build and Extend consume every shard's replica of the buffer: when one replica diverged, both refuse and leave
    every shard's lists and buffer as they were."""
    n = max(_counts(gpu))
    if n < 2:
        pytest.skip("needs 2 GPUs")
    rng = np.random.default_rng(35)
    X = rng.standard_normal((2600, DIM)).astype(np.float32)
    sx = gpu.ShardedIndex(n, gpu.IVF_FLAT, DIM, gpu.L2, nlist=20, m=8, k=K)
    sx.add(X[:2000])
    sx.build()
    before = [sx.shard(r)[0].lists() for r in range(n)]
    sx.add(X[2000:2500])
    sh0, _ = sx.shard(0)
    sh0.add(X[2500:])  # only shard 0's replica holds these rows
    for op in (sx.build, sx.extend):
        with pytest.raises(gpu._lib.PyropeGpuError) as e:
            op()
        assert e.value.code == gpu._lib.ERR_INVALID_STATE, e.value.message
        for r in range(n):
            sh, _ = sx.shard(r)
            off, rows, _ = sh.lists()
            np.testing.assert_array_equal(off, before[r][0], err_msg=f"{op.__name__}: shard {r} offsets")
            np.testing.assert_array_equal(rows, before[r][1], err_msg=f"{op.__name__}: shard {r} rows")
            assert sh.stats()["buffer"] == (600 if r == 0 else 500), f"{op.__name__}: shard {r} buffer"
            del sh
    del sh0
    sx.close()


# ---- Head+Tail with string ids: a CPU model of compaction by Extend ------------------------------------------------
class RefExtendDelta:
    """DeltaVectorIndex whose compaction is Extend, over the oracle: the head is an oracle FLAT index; the tail is kept
    as per-list entries [id, vector or code, dead] and handed to an oracle IVF index (live entries, list order)."""

    def __init__(self, kind, nlist, m):
        self.kind, self.nlist, self.m = kind, nlist, m
        self.head = orc.FlatIndex(DIM, orc.L2)
        self.head_rows, self.head_pos = [], {}
        self.lists = None
        self.where = {}  # id -> (list, position) of its current tail entry
        self.vec_of = {}  # id -> the vector its current tail entry was made from

    def add(self, i, v):
        self.head.upsert(i, v)
        if i in self.head_pos:
            self.head_rows[self.head_pos[i]] = (i, v)
        else:
            self.head_pos[i] = len(self.head_rows)
            self.head_rows.append((i, v))

    def delete(self, i):
        h = self.head.delete(i)
        if i in self.head_pos:
            self.head_rows[self.head_pos.pop(i)] = None
        t = False
        if self.kind == "ivf_flat" and i in self.where:  # IVF_PQ deletes only buffered rows
            c, j = self.where.pop(i)
            self.lists[c][j][2] = True
            self._adopt()
            t = True
        return h or t

    def _moved(self):
        out = [x for x in self.head_rows if x is not None]
        for i, _ in out:
            self.head.delete(i)
        self.head_rows, self.head_pos = [], {}
        return out

    def build(self):  # the first compaction: an oracle Build over the moved rows
        rows = self._moved()
        if self.kind == "ivf_flat":
            t = orc.IvfFlatIndex(DIM, orc.L2, nlist=self.nlist)
        else:
            t = orc.IvfPqIndex(DIM, orc.L2, m=self.m, k=K, nlist=self.nlist)
        vec = {}
        for i, v in rows:
            t.add(i, v)
            vec[i] = v
            self.vec_of[i] = v
        t.build()
        self.cent = t.centroids()
        self.lists = []
        if self.kind == "ivf_flat":
            for ids in t.lists():
                self.lists.append([[int(i), vec[int(i)], False] for i in ids])
        else:
            self.pq = orc.ProductQuantizer(DIM, self.m, K)
            self.pq.set_codebook(t.pq().codebook(), t.pq().ksub())
            self.cb = t.pq().codebook()
            for ids, codes in t.lists():
                self.lists.append([[int(i), c, False] for i, c in zip(ids, codes)])
        self.where = {e[0]: (c, j) for c, lst in enumerate(self.lists) for j, e in enumerate(lst)}
        self._adopt()

    def extend(self):
        for i, v in self._moved():
            if i in self.where:  # the shadowed entry becomes deleted
                c, j = self.where.pop(i)
                self.lists[c][j][2] = True
            a = orc.find_nearest_centroid(v, self.cent, orc.L2)
            payload = v if self.kind == "ivf_flat" else self.pq.encode((v - self.cent[a]).astype(np.float32))
            self.lists[a].append([i, payload, False])
            self.vec_of[i] = v
            self.where[i] = (a, len(self.lists[a]) - 1)
        self._adopt()

    def _adopt(self):
        off, ids, pay = [0], [], []
        for lst in self.lists:
            for e in lst:
                if not e[2]:
                    ids.append(e[0])
                    pay.append(e[1])
            off.append(len(ids))
        off = np.array(off, np.int64)
        ids = np.array(ids, np.int64)
        if self.kind == "ivf_flat":
            self.tail = orc.IvfFlatIndex(DIM, orc.L2, nlist=self.nlist)
            self.tail.adopt(self.cent, off, ids, np.array(pay, np.float32).reshape(-1, DIM))
        else:
            self.tail = orc.IvfPqIndex(DIM, orc.L2, m=self.m, k=K, nlist=self.nlist)
            self.tail.adopt(self.cent, self.cb, off, ids, np.array(pay, np.uint8).reshape(-1, self.m))

    def search(self, q, k, nprobe):
        return orc.delta_merge(self.head.search(q, k), self.tail.search(q, k, nprobe=nprobe), k)


def _check(ref, d, vi, Q, k, nprobe, ctx):
    got = d.SearchBatch(Q, k, vi.SearchOptions(NProbe=nprobe))
    for qi, g in zip(Q, got):
        rid, rsc = ref.search(qi, k, nprobe)
        assert_topk_equivalent(rid, rsc, [int(r.Id[1:]) for r in g], [r.Score for r in g], ctx=ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("tail_kind", ["ivf_flat", "ivf_pq"])
@pytest.mark.parametrize("devices", [None, "all"])
def test_delta_compaction_by_extend_matches_model(gpu, vi, tail_kind, devices):
    nlist, m = 12, 4
    devs = None if devices is None else _counts(gpu)[-1]
    rng = np.random.default_rng(44)
    base = rng.random((4000, DIM), dtype=np.float32)
    Q = rng.random((24, DIM), dtype=np.float32)
    if tail_kind == "ivf_flat":
        tail = vi.IvfFlatVectorIndex(DIM, vi.VectorMetric.L2, nList=nlist, devices=devs)
    else:
        tail = vi.IvfPqVectorIndex(DIM, vi.VectorMetric.L2, m=m, k=K, nList=nlist, devices=devs)
    if devs is not None:
        gpu._lib.check(gpu.load().pyrope_gpu_init(0))
    d = vi.DeltaVectorIndex(vi.BruteForceVectorIndex(DIM, vi.VectorMetric.L2), tail)
    ref = RefExtendDelta(tail_kind, nlist, m)
    d.Upsert("v0", base[0])
    ref.add(0, base[0])
    with pytest.raises(vi.InvalidOperationException):  # an unbuilt tail refuses before any row moves
        d.Extend()
    n0 = 1500
    for i in range(1, n0):
        ref.add(i, base[i])
        d.Upsert(f"v{i}", base[i])
    d.Build()
    ref.build()
    _check(ref, d, vi, Q, 10, 4, f"{tail_kind} after build")
    vb = vi.VectorIndexBatcher(d, max_batch=32, max_wait_us=2000)
    nxt = n0
    for rnd in range(4):
        for _ in range(400):
            op = rng.random()
            if op < 0.6:
                i = nxt
                nxt += 1
            else:
                i = int(rng.integers(0, nxt))
            if op < 0.85:
                v = base[i] if i < len(base) else rng.random(DIM, dtype=np.float32)
                if op >= 0.6:
                    v = rng.random(DIM, dtype=np.float32)
                ref.add(i, v)
                d.Upsert(f"v{i}", v)
            else:
                assert d.Delete(f"v{i}") == ref.delete(i), f"delete v{i}"
        _check(ref, d, vi, Q, 10, 4, f"{tail_kind} round {rnd} before extend")
        before = _wave(vb, Q)
        _same_wave(before, d.SearchBatch(Q, 10, vi.SearchOptions(NProbe=None)), f"round {rnd} batcher before")
        d.Extend()
        ref.extend()
        after = _wave(vb, Q)
        _same_wave(after, d.SearchBatch(Q, 10, vi.SearchOptions(NProbe=None)), f"round {rnd} batcher after")
        for nprobe in (1, 4, 12):
            _check(ref, d, vi, Q, 10, nprobe, f"{tail_kind} round {rnd} after extend nprobe={nprobe}")
    vb.close()
    # ids of the first compactions are still in the tail after the later ones (an IVF_PQ Build keeps only the last
    # compaction's rows): the model above holds them, and a search over every list finds them
    old = [i for i in range(n0, n0 + 200) if i in ref.where and not ref.head_pos.get(i)]
    assert len(old) > 50
    hits = d.SearchBatch(np.stack([ref_vec(ref, i) for i in old[:16]]), 10, vi.SearchOptions(NProbe=nlist))
    found = sum(any(r.Id == f"v{i}" for r in h) for i, h in zip(old[:16], hits))
    assert found >= (16 if tail_kind == "ivf_flat" else 8)
    d.close()
    tail.close()


def ref_vec(ref, i):
    """the vector the model's tail holds for id i (IVF_PQ: centroid + decoded code is not needed, the original row is
    kept next to it by _vec_of)"""
    return ref.vec_of[i]


def _wave(vb, Q):
    out = [None] * len(Q)

    def run(i):
        out[i] = vb.Search(Q[i], 10)

    th = [threading.Thread(target=run, args=(i,)) for i in range(len(Q))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    return out


def _same_wave(a, b, ctx):
    for q, (x, y) in enumerate(zip(a, b)):
        assert [r.Id for r in x] == [r.Id for r in y], f"{ctx} q{q}: ids"
        assert [r.Score for r in x] == [r.Score for r in y], f"{ctx} q{q}: scores"


@pytest.mark.gpu
@pytest.mark.parametrize("tail_kind", ["ivf_flat", "ivf_pq"])
def test_vindex_extend_ids_and_snapshot(gpu, vi, tail_kind, tmp_path):
    rng = np.random.default_rng(5)
    X = rng.random((2600, DIM), dtype=np.float32)
    mk = (lambda: vi.IvfFlatVectorIndex(DIM, vi.VectorMetric.L2, nList=10)) if tail_kind == "ivf_flat" else \
        (lambda: vi.IvfPqVectorIndex(DIM, vi.VectorMetric.L2, m=8, k=K, nList=10))
    a = mk()
    for i in range(2000):
        a.Add(f"a{i}", X[i])
    a.Build()
    for i in range(2000, 2600):
        a.Add(f"a{i}", X[i])
    a.Upsert("a3", X[3] + 0.5)  # an indexed id re-added: its list entry is shadowed until the Extend
    a.Extend()
    if tail_kind == "ivf_flat":
        assert a.GetStats().Count == 2600
        assert a.Delete("a2100") and not a.Delete("a2100")
    res = a.Search(X[2500], 10, vi.SearchOptions(NProbe=10))
    assert "a2500" in [r.Id for r in res]
    p = str(tmp_path / "leaf.bin")
    a.Snapshot(p)
    b = mk()
    b.Load(p)
    Q = rng.random((16, DIM), dtype=np.float32)
    for x, y in zip(a.SearchBatch(Q, 10), b.SearchBatch(Q, 10)):
        assert [r.Id for r in x] == [r.Id for r in y]
        assert [r.Score for r in x] == [r.Score for r in y]
    b.Upsert("a2200", X[7])  # an extended id behaves like a built one after the reload
    b.Extend()
    ids = [r.Id for r in b.Search(X[7], 10, vi.SearchOptions(NProbe=10))]
    assert "a2200" in ids and ids.count("a2200") == 1


def test_extend_null_handles_are_invalid_arg():
    from pyrope_b200 import _lib
    L = _lib.load()
    for fn in ("pyrope_index_extend", "pyrope_sharded_extend", "pyrope_delta_extend_tail", "pyrope_vindex_extend"):
        assert getattr(L, fn)(None) == _lib.ERR_INVALID_ARG, fn
