"""The reference's index classes, by their own names, over libpyrope_gpu.so (ctypes -> csrc/vindex.cu).

Same constructors, methods, argument meaning and error behaviour as
src/Pyrope.GarnetServer/Vector/{BruteForce,IvfFlat,IvfPq,Delta}VectorIndex.cs, so the parity tests read like
the reference's xunit tests.  All state (vectors, id dictionaries, tombstones, lists) lives in the native
library; this file only converts arguments and maps status codes to exception types.  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from enum import IntEnum

import numpy as np

from . import _lib
from ._lib import _np, _p, vp


class VectorMetric(IntEnum):  # IVectorIndex.cs:5-10
    L2 = 0
    InnerProduct = 1
    Cosine = 2


class ArgumentException(ValueError):
    pass


class ArgumentNullException(ArgumentException):
    pass


class ArgumentOutOfRangeException(ArgumentException):
    pass


class InvalidOperationException(RuntimeError):
    pass


@dataclass(frozen=True)
class SearchResult:  # IVectorIndex.cs:31
    Id: str
    Score: float


@dataclass(frozen=True)
class SearchOptions:  # IVectorIndex.cs:33-38
    MaxScans: int | None = None
    NProbe: int | None = None
    EfSearch: int | None = None  # HNSW only; ignored here as in the reference's IVF / FLAT classes


@dataclass(frozen=True)
class IndexStats:  # IVectorIndex.cs:40
    Count: int
    Dimension: int
    Metric: str


def _ck(rc: int):
    if rc != _lib.OK:
        _raise(rc)


def _raise_msg(rc: int, msg: str):
    if rc == _lib.ERR_INVALID_ARG:
        raise (ArgumentNullException if "cannot be null" in msg else ArgumentException)(msg)
    if rc == _lib.ERR_DIMENSION:
        raise ArgumentException(msg)  # "Vector dimension mismatch" => VEC_ERR_DIM (VectorCommandSet.cs:837-847)
    if rc == _lib.ERR_OUT_OF_RANGE:
        raise ArgumentOutOfRangeException(msg)
    if rc == _lib.ERR_INVALID_STATE:
        raise InvalidOperationException(msg)
    if rc == _lib.ERR_NOT_FOUND:
        raise FileNotFoundError(msg)
    raise _lib.PyropeGpuError(rc, msg)


def _raise(rc: int):
    _raise_msg(rc, (_lib.load().pyrope_last_error() or b"").decode("utf-8", "replace"))


def _id_string(ordinal: int) -> str:
    L = _lib.load()
    n = C.c_int32(0)
    _ck(L.pyrope_vindex_id(ordinal, None, 0, C.byref(n)))
    buf = C.create_string_buffer(n.value + 1)
    _ck(L.pyrope_vindex_id(ordinal, buf, n.value + 1, C.byref(n)))
    return buf.raw[:n.value].decode("utf-8")


def _id_strings(ordinals: np.ndarray) -> list[str]:
    """pyrope_vindex_ids: every id of a result list under one lock (empty slots, ordinal -1, give '')."""
    L = _lib.load()
    o = _np(ordinals, np.int64)
    n = o.size
    off = np.zeros(n + 1, np.int64)
    nbytes = C.c_int64(0)
    _ck(L.pyrope_vindex_ids(_p(o), n, None, 0, _p(off), C.byref(nbytes)))
    buf = C.create_string_buffer(max(1, nbytes.value))
    _ck(L.pyrope_vindex_ids(_p(o), n, buf, nbytes.value, _p(off), C.byref(nbytes)))
    raw = buf.raw
    return [raw[off[i]:off[i + 1]].decode("utf-8") for i in range(n)]


def _idb(id_):
    return None if id_ is None else str(id_).encode("utf-8")


def _options(options: SearchOptions | None):
    """(max_scans, nprobe) on the ABI.  null = no budget (-1); a caller's MaxScans <= 0 scans nothing in the reference
    and must not become "no budget"."""
    ms = -1 if options is None or options.MaxScans is None else max(int(options.MaxScans), 0)
    npb = -1 if options is None or options.NProbe is None else int(options.NProbe)
    return ms, npb


class _VectorIndex:
    """IVectorIndex (IVectorIndex.cs:14-29)."""

    _v = None

    def _vec(self, vector):
        if vector is None:
            return None, 0
        a = _np(vector, np.float32).reshape(-1)
        return a, a.size

    # ---- IVectorIndex
    @property
    def Dimension(self) -> int:
        return self._dim

    @property
    def Metric(self) -> VectorMetric:
        return self._metric

    def Add(self, id, vector):
        a, n = self._vec(vector)
        _ck(_lib.load().pyrope_vindex_add(self._v, _idb(id), _p(a), n))

    def Upsert(self, id, vector):
        a, n = self._vec(vector)
        _ck(_lib.load().pyrope_vindex_upsert(self._v, _idb(id), _p(a), n))

    def Delete(self, id) -> bool:
        out = C.c_int32(0)
        _ck(_lib.load().pyrope_vindex_delete(self._v, _idb(id), C.byref(out)))
        return bool(out.value)

    def Build(self):
        _ck(_lib.load().pyrope_vindex_build(self._v))

    def Search(self, query, topK: int, options: SearchOptions | None = None):
        res = self.SearchBatch([query] if query is not None else None, topK, options)
        return res[0]

    def SearchBatch(self, queries, topK: int, options: SearchOptions | None = None):
        """nq queries through one batched call (what the micro-batcher hands the library)."""
        if queries is None:
            Q, nq, ln = None, 1, 0
        else:
            Q = _np(queries, np.float32)
            if Q.ndim == 1:
                Q = Q[None, :]
            nq, ln = Q.shape
        kk = max(int(topK), 1)
        scores = np.zeros((nq, kk), np.float32)
        ids = np.full((nq, kk), -1, np.int64)
        counts = np.zeros(nq, np.int32)
        ms, npb = _options(options)
        _ck(_lib.load().pyrope_vindex_search(self._v, nq, _p(Q), ln, int(topK), ms, npb, _p(scores), _p(ids), _p(counts)))
        names = _id_strings(ids.reshape(-1))  # one call, one lock for the whole result list
        out = []
        for i in range(nq):
            out.append([SearchResult(names[i * kk + j], float(scores[i, j])) for j in range(int(counts[i]))])
        return out

    def Snapshot(self, path: str):
        _ck(_lib.load().pyrope_vindex_snapshot(self._v, _idb(path) if path is not None else None))

    def Load(self, path: str):
        _ck(_lib.load().pyrope_vindex_load(self._v, _idb(path) if path is not None else None))

    def GetStats(self) -> IndexStats:
        cnt, dim, met = C.c_int64(0), C.c_int32(0), C.c_int32(0)
        _ck(_lib.load().pyrope_vindex_stats(self._v, C.byref(cnt), C.byref(dim), C.byref(met)))
        return IndexStats(cnt.value, dim.value, VectorMetric(met.value).name)

    def GetCentroids(self):
        """ICentroidsProvider.GetCentroids: None until built (IvfFlatVectorIndex.cs:314-325)."""
        n = C.c_int32(0)
        _ck(_lib.load().pyrope_vindex_get_centroids(self._v, None, C.byref(n)))
        if n.value == 0:
            return None
        out = np.zeros((n.value, self._dim), np.float32)
        _ck(_lib.load().pyrope_vindex_get_centroids(self._v, _p(out), C.byref(n)))
        return [out[i] for i in range(n.value)]

    def close(self):
        if getattr(self, "_v", None):
            _lib.load().pyrope_vindex_destroy(self._v)
            self._v = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Extendable:
    """Extend() of the IVF leaves and the Head+Tail (pyrope_vindex_extend; no counterpart in the reference): the write
    buffer joins the built inverted lists without re-training.  On a DeltaVectorIndex it compacts the head into the tail
    that way.  Not built -> InvalidOperationException."""

    def Extend(self):
        _ck(_lib.load().pyrope_vindex_extend(self._v))


class _BorrowedGpuIndex(_lib.GpuIndex):
    """Row-ordinal view of a handle the vindex owns: never destroys it."""

    def close(self):
        self._h = None

    __del__ = close


def _devices(devices):
    """None -> one device; an int N -> devices 0..N-1; a sequence -> those CUDA ordinals."""
    if devices is None:
        return None
    if isinstance(devices, (int, np.integer)):
        return list(range(int(devices)))
    return [int(d) for d in devices]


class _Leaf(_VectorIndex):
    def _create(self, kind, dimension, metric, nlist=100, m=4, k=256, devices=None):
        v = vp()
        devs = _devices(devices)
        if devs is None:
            _ck(_lib.load().pyrope_vindex_create(kind, int(dimension), int(metric), int(nlist), int(m), int(k), C.byref(v)))
        else:  # the same index over several GPUs of the box (pyrope_sharded_*)
            dv = np.asarray(devs, np.int32)
            _ck(_lib.load().pyrope_vindex_create_sharded(len(devs), dv.ctypes.data_as(_lib.i32p), kind, int(dimension),
                                                         int(metric), int(nlist), int(m), int(k), C.byref(v)))
        self._v, self._dim, self._metric = v, int(dimension), VectorMetric(int(metric))
        self._devices = devs

    def native(self) -> _lib.GpuIndex:
        """Row-ordinal view of the same index (borrowed handle) for bit-exact parity reads."""
        h = vp()
        _ck(_lib.load().pyrope_vindex_native(self._v, C.byref(h)))
        if not h.value:
            raise InvalidOperationException("a sharded index has no single row-ordinal handle")
        g = _BorrowedGpuIndex.__new__(_BorrowedGpuIndex)
        g._h, g.kind, g.dim, g.metric = h, self._kind, self._dim, int(self._metric)
        g.nlist, g.m, g.k = self._nlist, self._m, self._k
        g._owner = self  # keep the owning index alive while the view is in use
        return g


class BruteForceVectorIndex(_Leaf):
    """BruteForceVectorIndex(dimension, metric) — BruteForceVectorIndex.cs:42-51."""

    def __init__(self, dimension: int, metric: VectorMetric = VectorMetric.L2):
        self._kind, self._nlist, self._m, self._k = _lib.FLAT, 0, 0, 0
        self._create(_lib.FLAT, dimension, metric)
        self._quant = False

    @property
    def EnableQuantization(self) -> bool:  # BruteForceVectorIndex.cs:36-40
        return self._quant

    @EnableQuantization.setter
    def EnableQuantization(self, value: bool):
        _ck(_lib.load().pyrope_vindex_set_quantization(self._v, 1 if value else 0))
        self._quant = bool(value)


class IvfFlatVectorIndex(_Extendable, _Leaf):
    """IvfFlatVectorIndex(dimension, metric, nList = 100) — IvfFlatVectorIndex.cs:27-33.  devices (N or a list of CUDA
    ordinals) shards the inverted lists over those GPUs; results equal the one-device index's."""

    def __init__(self, dimension: int, metric: VectorMetric = VectorMetric.L2, nList: int = 100, devices=None):
        self._kind, self._nlist, self._m, self._k = _lib.IVF_FLAT, nList, 0, 0
        self._create(_lib.IVF_FLAT, dimension, metric, nlist=nList, devices=devices)


class IvfPqVectorIndex(_Extendable, _Leaf):
    """IvfPqVectorIndex(dimension, metric, m, k = 256, nList = 100) — IvfPqVectorIndex.cs:27-35.  devices as for
    IvfFlatVectorIndex."""

    def __init__(self, dimension: int, metric: VectorMetric = VectorMetric.L2, m: int = 4, k: int = 256,
                 nList: int = 100, devices=None):
        self._kind, self._nlist, self._m, self._k = _lib.IVF_PQ, nList, m, k
        self._create(_lib.IVF_PQ, dimension, metric, nlist=nList, m=m, k=k, devices=devices)


class DeltaVectorIndex(_Extendable, _VectorIndex):
    """DeltaVectorIndex(head, tail) — DeltaVectorIndex.cs:18-28; Search merges on the device, Build compacts
    head -> tail device-to-device."""

    def __init__(self, head: _Leaf, tail: _Leaf):
        v = vp()
        _ck(_lib.load().pyrope_vindex_create_delta(head._v, tail._v, C.byref(v)))
        self._v, self._dim, self._metric = v, head.Dimension, head.Metric
        self._head, self._tail = head, tail  # keep both alive for as long as the delta borrows them


def create_index(algorithm: str | None, dimension: int, metric: VectorMetric, params: dict | None = None):
    """VectorIndexRegistry.IndexState..ctor (Services/VectorIndexRegistry.cs:81-113): a BruteForce head over the
    tail the Algorithm string names (default IVF_FLAT; m 4 / k 256 / nlist 100).  params["devices"] (N, or a list
    of CUDA ordinals) shards the tail over those GPUs and makes the first of them current for the head; a FLAT tail
    cannot be sharded (PyropeGpuError, UNSUPPORTED)."""
    params = params or {}
    algo = (algorithm or "IVF_FLAT").upper().replace("GPU_", "")
    devs = _devices(params.get("devices"))
    if algo == "IVF_PQ":
        tail = IvfPqVectorIndex(dimension, metric, int(params.get("m", 4)), int(params.get("k", 256)),
                                int(params.get("nlist", 100)), devices=devs)
    elif algo == "FLAT":
        if devs is not None:
            raise _lib.PyropeGpuError(_lib.ERR_UNSUPPORTED, "a FLAT tail cannot be sharded over devices")
        tail = BruteForceVectorIndex(dimension, metric)
    else:
        tail = IvfFlatVectorIndex(dimension, metric, int(params.get("nlist", 100)), devices=devs)
    if devs is not None:  # the head lives on the tail's first device
        _ck(_lib.load().pyrope_gpu_init(devs[0]))
    return DeltaVectorIndex(BruteForceVectorIndex(dimension, metric), tail)


class VectorIndexBatcher:
    """The Search of the C# shim in front of a micro-batcher (pyrope_batcher_create_vindex): each call enqueues one
    query and blocks while the dispatcher thread searches it together with the other callers' queries, then turns the
    id ordinals into strings.  A shim does that translation under the read lock its Search runs under, so an id in the
    result cannot be deleted and recycled before it is named.  Destroy the batcher (close) before the index."""

    def __init__(self, index: _VectorIndex, max_batch: int = 256, max_wait_us: int = 200):
        self._index = index
        self._b = _lib.Batcher(index, max_batch, max_wait_us)

    def Search(self, query, topK: int, options: SearchOptions | None = None) -> list[SearchResult]:
        if query is None:
            raise ArgumentNullException("Value cannot be null. (Parameter 'vector')")
        q = _np(query, np.float32).reshape(-1)
        if q.size != self._index.Dimension:  # ValidateDim: the batcher reads Dimension floats
            raise ArgumentException("Vector dimension mismatch")
        ms, npb = _options(options)
        kk = max(int(topK), 1)
        scores, ids, cnt = np.zeros(kk, np.float32), np.full(kk, -1, np.int64), C.c_int32(0)
        _ck(_lib.load().pyrope_batcher_search(self._b._b, _p(q), int(topK), ms, npb, _p(scores), _p(ids), C.byref(cnt)))
        n = cnt.value
        names = _id_strings(ids[:n]) if n else []
        return [SearchResult(names[j], float(scores[j])) for j in range(n)]

    def stats(self) -> dict:
        return self._b.stats()

    def close(self):
        self._b.close()
