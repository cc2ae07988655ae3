"""The micro-batcher in front of the objects a server holds (csrc/batcher.cu): a one-device index, a sharded index, a
Head+Tail (pyrope_delta) and a string-id index (pyrope_vindex), with callers of different topK sharing one batched
search, and the per-query k of the Head+Tail merge (pyrope_delta_search_batch_topk) that makes that exact."""
import ctypes as C
import threading

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.parity import assert_topk_equivalent
from tests.test_gpu_vector_index import RefDelta

gpu_only = pytest.mark.gpu
DIM = 32


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


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


# ---------------------------------------------------------------------------------------------- raw Head+Tail handles
def _delta(gpu, head, tail):
    d = C.c_void_p()
    L = gpu.load()
    if isinstance(tail, gpu.ShardedIndex):
        gpu._lib.check(L.pyrope_delta_create_sharded(head._h, tail._s, C.byref(d)))
    else:
        gpu._lib.check(L.pyrope_delta_create(head._h, tail._h, C.byref(d)))
    return d


def _dsearch(gpu, d, Q, k, max_scans=-1, nprobe=-1):
    nq = len(Q)
    S, R, N = np.zeros((nq, k), np.float32), np.full((nq, k), -1, np.int64), np.zeros(nq, np.int32)
    gpu._lib.check(gpu.load().pyrope_delta_search_batch(d, nq, _p(Q), k, max_scans, nprobe, _p(S), _p(R), _p(N)))
    return S, R, N


def _dsearch_topk(gpu, d, Q, topks, max_scans=-1, nprobe=-1):
    nq, kk = len(Q), int(max(topks))
    t = np.ascontiguousarray(topks, np.int32)
    S, R, N = np.zeros((nq, kk), np.float32), np.full((nq, kk), -1, np.int64), np.zeros(nq, np.int32)
    gpu._lib.check(gpu.load().pyrope_delta_search_batch_topk(d, nq, _p(Q), _p(t), max_scans, nprobe, _p(S), _p(R), _p(N)))
    return S, R, N


def _make_tail(gpu, kind, n_dev):
    kw = dict(nlist=16, m=8, k=64)
    return gpu.ShardedIndex(n_dev, kind, DIM, gpu.L2, **kw) if n_dev else gpu.GpuIndex(kind, DIM, gpu.L2, **kw)


def _head_tail(gpu, kind, n_dev, head_rows, nprobe):
    """A built tail of 6,000 rows (labels 0..5999) and a FLAT head of head_rows rows far from every query.  For each of the
    48 queries the head also holds the tail's best id at distance 3 from the query: the head's best row, but worse than
    the tail's 100th.  So with topK = k the tail's copy is de-duplicated away and the head's copy takes the k-th place,
    where a search at a larger K cut after the merge would put the tail's (k+1)-th."""
    rng = np.random.default_rng(7)
    X = rng.random((6000, DIM), dtype=np.float32)
    Q = (X[:48] + 0.01 * rng.random((48, DIM), dtype=np.float32)).astype(np.float32)
    tail = _make_tail(gpu, kind, n_dev)
    tail.add(X, labels=np.arange(6000, dtype=np.int64))
    tail.build()
    _, best, _ = tail.search(Q, 1, nprobe=nprobe)
    head = gpu.GpuIndex(gpu.FLAT, DIM, gpu.L2)
    head.add(rng.random((head_rows, DIM), dtype=np.float32) + 5.0, labels=np.arange(head_rows, dtype=np.int64) + 1_000_000)
    near = Q.copy()
    near[:, 0] += 3.0
    head.add(near, labels=best[:, 0].copy())
    return head, tail, Q


def _compare_topk(gpu, d, Q, topks, nprobe, exact, ctx):
    got = _dsearch_topk(gpu, d, Q, topks, nprobe=nprobe)
    for t in sorted(set(int(x) for x in topks)):
        ref = _dsearch(gpu, d, Q, t, nprobe=nprobe)
        for i in np.nonzero(np.asarray(topks) == t)[0]:
            c = int(ref[2][i])
            assert int(got[2][i]) == c, f"{ctx} q{i} k={t}: count {int(got[2][i])} != {c}"
            if exact:
                np.testing.assert_array_equal(got[1][i][:c], ref[1][i][:c], err_msg=f"{ctx} q{i} k={t}: ids")
                assert got[0][i][:c].tobytes() == ref[0][i][:c].tobytes(), f"{ctx} q{i} k={t}: score bits"
            else:
                assert_topk_equivalent(ref[1][i][:c], ref[0][i][:c], got[1][i][:c], got[0][i][:c], ctx=f"{ctx} q{i} k={t}")
    return got


@gpu_only
@pytest.mark.parametrize("head_rows", [500, 9000])  # below / above the FLAT tensor-core path's 8,192 rows
def test_per_query_k_merge_is_bit_exact(gpu, head_rows):
    rng = np.random.default_rng(11)
    for kind in (gpu.IVF_FLAT, gpu.IVF_PQ):
        for n_dev in [0] + _counts(gpu):  # 0: a one-device tail, else a tail sharded over n_dev devices
            head, tail, Q = _head_tail(gpu, kind, n_dev, head_rows, nprobe=4)
            d = _delta(gpu, head, tail)
            try:
                ctx = f"kind={kind} devices={n_dev} head={head_rows}"
                topks = rng.integers(1, 101, len(Q)).astype(np.int32)
                topks[:4] = [1, 2, 3, 100]
                # every topK in 1..100 selects the same kernels as 100 (the tensor-core FLAT path takes k + margin <= 224)
                _compare_topk(gpu, d, Q, topks, 4, True, ctx)
                # the construction bites: cutting the merge at K after the fact would differ for some query
                full = _dsearch(gpu, d, Q, int(topks.max()), nprobe=4)
                own = _dsearch(gpu, d, Q, 3, nprobe=4)
                i = 2  # topK 3
                assert list(full[1][i][:3]) != list(own[1][i][:int(own[2][i])]), f"{ctx}: truncation after the merge not exercised"
                if head_rows > 8192:
                    # K = 200 takes the CUDA-core FLAT scan for the head, k <= 100 the tensor cores: the parity bar applies
                    mixed = topks.copy()
                    mixed[4] = 200
                    _compare_topk(gpu, d, Q, mixed, 4, False, ctx + " K=200")
            finally:
                gpu.load().pyrope_delta_destroy(d)
            if n_dev:
                tail.close()


# ---------------------------------------------------------------------------------------------- deterministic coalescing
def _wave(search, n):
    out = [None] * n

    def run(i):
        try:
            out[i] = search(i)
        except Exception as e:  # noqa: BLE001 - handed back to the test
            out[i] = e

    th = [threading.Thread(target=run, args=(i,)) for i in range(n)]
    [t.start() for t in th]
    [t.join() for t in th]
    return out


CASES = [  # (topKs, MaxScans per caller, batches)
    ([9, 12, 16], [-1, -1, -1], 1),
    ([9, 40], [-1, -1], 2),
    ([10, 10], [-1, 300], 2),
]


def _groups(topks, scans):
    g = {}
    for i, (t, s) in enumerate(zip(topks, scans)):
        c = 1 << (int(t) - 1).bit_length()
        g.setdefault((c, s), []).append(i)
    return list(g.values())


def _check_row_target(gpu, target, direct, Q, ctx):
    """target: GpuIndex / ShardedIndex / raw delta; direct(Qg, topk, max_scans) -> (scores, rows, counts) or raises"""
    for topks, scans, nb in CASES:
        b = gpu.Batcher(target, max_batch=len(topks), max_wait_us=1_000_000)
        try:
            got = _wave(lambda i: b.search(Q[i], topks[i], max_scans=scans[i], nprobe=4), len(topks))
            assert b.stats()["batches"] == nb, f"{ctx} {topks} {scans}: {b.stats()}"
        finally:
            b.close()
        for grp in _groups(topks, scans):
            Qg = Q[grp]
            for j, i in enumerate(grp):
                try:
                    s, r, c = direct(Qg, topks[i], scans[i])
                except gpu.PyropeGpuError as e:
                    assert isinstance(got[i], gpu.PyropeGpuError) and got[i].code == e.code, f"{ctx} caller {i}: {got[i]!r}"
                    continue
                assert not isinstance(got[i], Exception), f"{ctx} caller {i}: {got[i]!r}"
                gs, gr = got[i]
                n = int(c[j])
                np.testing.assert_array_equal(gr, r[j][:n], err_msg=f"{ctx} caller {i} ids")
                assert gs.tobytes() == s[j][:n].tobytes(), f"{ctx} caller {i} score bits"


@gpu_only
def test_coalescing_is_deterministic_on_row_targets(gpu):
    head, tail, Q = _head_tail(gpu, gpu.IVF_FLAT, 0, 500, nprobe=4)
    _check_row_target(gpu, tail, lambda Qg, k, ms: tail.search(Qg, k, max_scans=ms, nprobe=4), Q, "index")
    d = _delta(gpu, head, tail)
    try:
        _check_row_target(gpu, d, lambda Qg, k, ms: _dsearch(gpu, d, Qg, k, max_scans=ms, nprobe=4), Q, "delta")
    finally:
        gpu.load().pyrope_delta_destroy(d)
    for n in _counts(gpu):
        h2, sx, Q2 = _head_tail(gpu, gpu.IVF_PQ, n, 500, nprobe=4)
        _check_row_target(gpu, sx, lambda Qg, k, ms: sx.search(Qg, k, max_scans=ms, nprobe=4), Q2, f"sharded n={n}")
        d = _delta(gpu, h2, sx)
        try:
            _check_row_target(gpu, d, lambda Qg, k, ms: _dsearch(gpu, d, Qg, k, max_scans=ms, nprobe=4), Q2,
                              f"sharded delta n={n}")
        finally:
            gpu.load().pyrope_delta_destroy(d)
        sx.close()


def _string_delta(vi, n_dev, kind="IVF_FLAT", n0=1500, seed=3):
    rng = np.random.default_rng(seed)
    X = rng.random((n0 + 300, 16), dtype=np.float32)
    params = {"nlist": 12, "m": 4, "k": 64}
    if n_dev:
        params["devices"] = n_dev
    d = vi.create_index(kind, 16, vi.VectorMetric.L2, params)
    for i in range(n0):
        d.Upsert(f"v{i}", X[i])
    d.Build()
    for i in range(n0, n0 + 300):
        d.Upsert(f"v{i}", X[i])
    return d, X


@gpu_only
def test_coalescing_is_deterministic_on_string_id_head_tail(gpu, vi):
    for n_dev in [0] + _counts(gpu):
        d, X = _string_delta(vi, n_dev)
        Q = X[:3] + 0.01
        for topks, scans, nb in CASES:
            vb = vi.VectorIndexBatcher(d, max_batch=len(topks), max_wait_us=1_000_000)
            try:
                opts = [vi.SearchOptions(MaxScans=None if s < 0 else s, NProbe=4) for s in scans]
                got = _wave(lambda i: vb.Search(Q[i], topks[i], opts[i]), len(topks))
                assert vb.stats()["batches"] == nb
            finally:
                vb.close()
            for grp in _groups(topks, scans):
                for j, i in enumerate(grp):
                    try:
                        ref = d.SearchBatch(Q[grp], topks[i], opts[i])[j]
                    except gpu.PyropeGpuError as e:  # MaxScans on an IVF_FLAT tail over several devices
                        assert isinstance(got[i], gpu.PyropeGpuError) and got[i].code == e.code, f"caller {i}: {got[i]!r}"
                        continue
                    assert not isinstance(got[i], Exception), f"devices={n_dev} caller {i}: {got[i]!r}"
                    assert [r.Id for r in got[i]] == [r.Id for r in ref], f"devices={n_dev} {topks} caller {i}"
                    assert [r.Score for r in got[i]] == [r.Score for r in ref], f"devices={n_dev} {topks} caller {i}"
        d.close()


# ---------------------------------------------------------------------------------------------- against the oracle
@gpu_only
def test_concurrent_callers_match_the_oracle(gpu, vi):
    dim, n0 = 16, 1500
    rng = np.random.default_rng(11)
    base = rng.random((n0 + 400, dim), dtype=np.float32)
    Q = rng.random((256, dim), dtype=np.float32)
    rt = orc.IvfFlatIndex(dim, orc.L2, nlist=12)
    ref = RefDelta(dim, orc.L2, rt)
    d = vi.DeltaVectorIndex(vi.BruteForceVectorIndex(dim, vi.VectorMetric.L2), vi.IvfFlatVectorIndex(dim, vi.VectorMetric.L2, nList=12))
    for i in range(n0):
        ref.add(i, base[i])
        d.Upsert(f"v{i}", base[i])
    ref.build()
    d.Build()
    for i in range(n0, n0 + 300):
        ref.add(i, base[i])
        d.Upsert(f"v{i}", base[i])
    for j, i in enumerate(range(0, n0, 25)):  # ids the head now overrides
        ref.add(i, base[n0 + 300 + j])
        d.Upsert(f"v{i}", base[n0 + 300 + j])
    mix = [1, 5, 10, 20, 50, 100]
    vb = vi.VectorIndexBatcher(d, max_batch=64, max_wait_us=2000)
    out = [None] * len(Q)

    def worker(t):
        for i in range(t * 8, t * 8 + 8):
            ms = None if i % 2 == 0 else 300
            out[i] = vb.Search(Q[i], mix[i % len(mix)], vi.SearchOptions(MaxScans=ms, NProbe=4))

    th = [threading.Thread(target=worker, args=(t,)) for t in range(32)]
    [t.start() for t in th]
    [t.join() for t in th]
    st = vb.stats()
    vb.close()
    assert st["queries"] == len(Q) and st["batches"] < len(Q)
    for i in range(len(Q)):
        kw = {"nprobe": 4} if i % 2 == 0 else {"nprobe": 4, "max_scans": 300}
        rid, rsc = ref.search(Q[i], mix[i % len(mix)], **kw)
        ids = [r.Id for r in out[i]]
        by_name = {f"v{int(x)}": int(x) for x in rid}
        assert all(s.startswith("v") for s in ids)
        assert set(ids) <= set(by_name) | {f"v{j}" for j in range(n0 + 400)}, f"caller {i}: unknown id"
        assert_topk_equivalent([by_name[f"v{int(x)}"] for x in rid], rsc, [int(s[1:]) for s in ids],
                               [r.Score for r in out[i]], ctx=f"caller {i}")


# ---------------------------------------------------------------------------------------------- per-caller errors
@gpu_only
def test_errors_stay_with_their_caller(gpu):
    head, tail, Q = _head_tail(gpu, gpu.IVF_FLAT, 0, 500, nprobe=4)
    d = _delta(gpu, head, tail)
    try:
        for target, bad, code in ((d, 0, gpu._lib.ERR_OUT_OF_RANGE), (tail, 0, None)):
            b = gpu.Batcher(target, max_batch=2, max_wait_us=1_000_000)   # the two good callers (one topK class) fill the batch
            topks = [10, 12, bad]
            got = _wave(lambda i: b.search(Q[i], topks[i], nprobe=4), 3)
            assert b.stats() == {"batches": 1, "queries": 2}
            b.close()
            assert all(not isinstance(g, Exception) and len(g[1]) == k for g, k in zip(got[:2], topks[:2]))
            if code is None:                                              # topK 0 on an IVF leaf: an empty result
                assert not isinstance(got[2], Exception) and len(got[2][1]) == 0
            else:
                assert isinstance(got[2], gpu.PyropeGpuError) and got[2].code == code
                assert "topK must be positive" in str(got[2])             # pyrope_batcher_last_error
    finally:
        gpu.load().pyrope_delta_destroy(d)
    for n in _counts(gpu):
        sx = _make_tail(gpu, gpu.IVF_PQ, n)
        rng = np.random.default_rng(1)
        sx.add(rng.random((3000, DIM), dtype=np.float32))
        sx.build()
        lim = min(1024, 4096 // n)
        with pytest.raises(gpu.PyropeGpuError) as direct:
            sx.search(Q[:1], lim + 1, nprobe=4)
        b = gpu.Batcher(sx, max_batch=2, max_wait_us=1_000_000)
        topks = [10, lim, lim + 1]
        got = _wave(lambda i: b.search(Q[i], topks[i], nprobe=4), 3)
        b.close()
        assert not isinstance(got[0], Exception) and len(got[0][1]) == 10
        assert not isinstance(got[1], Exception) and len(got[1][1]) == int(sx.search(Q[1:2], lim, nprobe=4)[2][0])
        assert isinstance(got[2], gpu.PyropeGpuError) and got[2].code == direct.value.code == gpu._lib.ERR_UNSUPPORTED
        assert "topK" in str(got[2])
        sx.close()


# ---------------------------------------------------------------------------------------------- writes between waves
class _RWLock:
    """The shim's ReaderWriterLockSlim: Search under the read lock, writes under the write lock."""

    def __init__(self):
        self._c, self._readers, self._writer = threading.Condition(), 0, False

    def read(self):
        lock = self

        class _R:
            def __enter__(self):
                with lock._c:
                    lock._c.wait_for(lambda: not lock._writer)
                    lock._readers += 1

            def __exit__(self, *a):
                with lock._c:
                    lock._readers -= 1
                    lock._c.notify_all()
        return _R()

    def write(self):
        lock = self

        class _W:
            def __enter__(self):
                with lock._c:
                    lock._c.wait_for(lambda: not lock._writer and lock._readers == 0)
                    lock._writer = True

            def __exit__(self, *a):
                with lock._c:
                    lock._writer = False
                    lock._c.notify_all()
        return _W()


@gpu_only
def test_writes_between_waves(gpu, vi):
    d, X = _string_delta(vi, 0, seed=9)
    rng = np.random.default_rng(9)
    rw = _RWLock()
    vb = vi.VectorIndexBatcher(d, max_batch=16, max_wait_us=1_000_000)
    opts = vi.SearchOptions(NProbe=4)
    deleted = set()
    try:
        for wave in range(4):
            Q = X[rng.integers(0, len(X), 16)] + 0.001
            topks = [5 + (i % 4) for i in range(16)]                       # one topK class: one batch per wave

            def search(i):
                with rw.read():
                    return vb.Search(Q[i], topks[i], opts)

            got = _wave(search, 16)
            with rw.read():
                for i in range(16):
                    ref = d.SearchBatch(Q, topks[i], opts)[i]
                    assert [(r.Id, r.Score) for r in got[i]] == [(r.Id, r.Score) for r in ref], f"wave {wave} caller {i}"
                    assert not deleted & {r.Id for r in got[i]}, f"wave {wave}: a deleted id came back"
            with rw.write():                                               # Upsert / Delete / Build between waves
                for i in rng.integers(0, len(X), 40):
                    if f"v{i}" in deleted:
                        continue
                    d.Upsert(f"v{i}", rng.random(16, dtype=np.float32))
                for i in rng.integers(0, len(X), 20):
                    if d.Delete(f"v{i}"):
                        deleted.add(f"v{i}")
                if wave % 2 == 1:
                    d.Build()
    finally:
        vb.close()
    d.close()


# ---------------------------------------------------------------------------------------------- CPU
def test_new_batcher_targets_validate_before_cuda():
    from pyrope_b200 import _lib
    L = _lib.load()
    b = C.c_void_p()
    for fn in (L.pyrope_batcher_create_sharded, L.pyrope_batcher_create_delta, L.pyrope_batcher_create_vindex):
        assert fn(None, 8, 100, C.byref(b)) == _lib.ERR_INVALID_ARG
        assert L.pyrope_batcher_last_error()
    assert L.pyrope_batcher_create(None, 8, 100, C.byref(b)) == _lib.ERR_INVALID_ARG
