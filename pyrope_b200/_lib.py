"""ctypes binding of libpyrope_gpu.so (the C ABI in include/pyrope_gpu.h).

There is no CPU fallback: if the CUDA library is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpyrope_gpu.so")

FLAT, IVF_FLAT, IVF_PQ = 0, 1, 2
L2, INNER_PRODUCT, COSINE = 0, 1, 2

OK = 0
ERR_INVALID_ARG, ERR_DIMENSION, ERR_OUT_OF_RANGE, ERR_INVALID_STATE = -1, -2, -3, -4
ERR_NOT_FOUND, ERR_CUDA, ERR_OOM, ERR_UNSUPPORTED = -5, -6, -7, -8


class PyropeGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[{code}] {msg}")
        self.code = code
        self.message = msg


f32p = C.POINTER(C.c_float)
i64p = C.POINTER(C.c_int64)
i32p = C.POINTER(C.c_int32)
u8p = C.POINTER(C.c_uint8)
vp = C.c_void_p

# name -> (restype, argtypes): exactly the symbols include/pyrope_gpu.h declares
SIGNATURES = {
    "pyrope_gpu_init": (C.c_int, [C.c_int]),
    "pyrope_gpu_shutdown": (C.c_int, []),
    "pyrope_gpu_device_count": (C.c_int, [i32p]),
    "pyrope_last_error": (C.c_char_p, []),
    "pyrope_version": (C.c_int, []),
    "pyrope_index_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "pyrope_index_destroy": (C.c_int, [vp]),
    "pyrope_index_reserve": (C.c_int, [vp, C.c_int64]),
    "pyrope_index_add_batch": (C.c_int, [vp, C.c_int64, vp, vp, i64p]),
    "pyrope_index_add_batch_device": (C.c_int, [vp, C.c_int64, vp, vp, i64p]),
    "pyrope_index_update_row": (C.c_int, [vp, C.c_int64, vp]),
    "pyrope_index_delete_row": (C.c_int, [vp, C.c_int64]),
    "pyrope_index_shadow_row": (C.c_int, [vp, C.c_int64, C.c_int]),
    "pyrope_index_set_labels": (C.c_int, [vp, C.c_int64, vp]),
    "pyrope_index_set_quantization": (C.c_int, [vp, C.c_int]),
    "pyrope_index_build": (C.c_int, [vp]),
    "pyrope_index_extend": (C.c_int, [vp]),
    "pyrope_index_set_train_params": (C.c_int, [vp, C.c_int64, C.c_int]),
    "pyrope_index_set_codebooks": (C.c_int, [vp, C.c_int, vp, vp]),
    "pyrope_index_set_shard": (C.c_int, [vp, C.c_int, C.c_int]),
    "pyrope_index_threshold_exchange_handle": (C.c_int, [vp, C.c_int64, vp]),
    "pyrope_index_threshold_exchange_open": (C.c_int, [vp, C.c_int, C.c_int, vp]),
    "pyrope_index_threshold_exchange_close": (C.c_int, [vp]),
    "pyrope_index_threshold_exchange_epoch": (C.c_int, [vp, C.c_uint32]),
    "pyrope_index_threshold_exchange_array": (C.c_int, [vp, C.c_int64, C.POINTER(vp)]),
    "pyrope_index_threshold_exchange_attach": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(vp)]),
    "pyrope_topk_merge_dedupe_device": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, C.c_int, vp]),
    "pyrope_sharded_create": (C.c_int, [C.c_int, i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "pyrope_sharded_destroy": (C.c_int, [vp]),
    "pyrope_sharded_device_count": (C.c_int, [vp, i32p]),
    "pyrope_sharded_shard": (C.c_int, [vp, C.c_int, C.POINTER(vp), i32p]),
    "pyrope_sharded_note_rows": (C.c_int, [vp, C.c_int64]),
    "pyrope_sharded_set_train_params": (C.c_int, [vp, C.c_int64, C.c_int]),
    "pyrope_sharded_set_codebooks": (C.c_int, [vp, C.c_int, vp, vp]),
    "pyrope_sharded_add_batch": (C.c_int, [vp, C.c_int64, vp, vp, i64p]),
    "pyrope_sharded_delete_row": (C.c_int, [vp, C.c_int64]),
    "pyrope_sharded_update_row": (C.c_int, [vp, C.c_int64, vp]),
    "pyrope_sharded_shadow_row": (C.c_int, [vp, C.c_int64, C.c_int]),
    "pyrope_sharded_set_labels": (C.c_int, [vp, C.c_int64, vp]),
    "pyrope_sharded_is_built": (C.c_int, [vp, i32p]),
    "pyrope_sharded_get_centroids": (C.c_int, [vp, vp, i32p]),
    "pyrope_sharded_get_codebooks": (C.c_int, [vp, vp, vp]),
    "pyrope_sharded_snapshot": (C.c_int, [vp, C.c_char_p]),
    "pyrope_sharded_load": (C.c_int, [vp, C.c_char_p]),
    "pyrope_sharded_build": (C.c_int, [vp]),
    "pyrope_sharded_extend": (C.c_int, [vp]),
    "pyrope_sharded_stats": (C.c_int, [vp, i64p]),
    "pyrope_sharded_search_batch": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int64, C.c_int, vp, vp, vp]),
    "pyrope_sharded_search_batch_device": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int64, C.c_int, vp, vp, vp]),
    "pyrope_sharded_last_search_ms": (C.c_int, [vp, f32p]),
    "pyrope_sharded_last_error": (C.c_char_p, []),
    "pyrope_peer_group_create": (C.c_int, [C.c_int, C.c_int, C.c_size_t, C.c_int, C.POINTER(vp)]),
    "pyrope_peer_group_destroy": (C.c_int, [vp]),
    "pyrope_peer_group_handle": (C.c_int, [vp, vp]),
    "pyrope_peer_group_open": (C.c_int, [vp, vp]),
    "pyrope_peer_group_buffer": (C.c_int, [vp, C.POINTER(vp)]),
    "pyrope_peer_group_attach": (C.c_int, [vp, C.POINTER(vp)]),
    "pyrope_peer_allgather_device": (C.c_int, [vp, C.c_int, vp, C.c_size_t, C.POINTER(vp), vp]),
    "pyrope_peer_last_error": (C.c_char_p, []),
    "pyrope_index_is_built": (C.c_int, [vp, i32p]),
    "pyrope_index_get_centroids": (C.c_int, [vp, vp, i32p]),
    "pyrope_index_get_codebooks": (C.c_int, [vp, vp, vp]),
    "pyrope_index_get_lists": (C.c_int, [vp, vp, vp, vp, i64p]),
    "pyrope_index_snapshot": (C.c_int, [vp, C.c_char_p]),
    "pyrope_index_load": (C.c_int, [vp, C.c_char_p]),
    "pyrope_index_stats": (C.c_int, [vp, i64p, i64p, i32p, i32p]),
    "pyrope_index_search_batch": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int64, C.c_int, vp, vp, vp]),
    "pyrope_index_search_batch_device": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int64, C.c_int, vp, vp, vp, vp]),
    "pyrope_index_coarse_probe_device": (C.c_int, [vp, C.c_int64, vp, C.c_int, vp, vp]),
    "pyrope_index_search_batch_probed_device": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int64, C.c_int, vp, vp, vp, vp, vp]),
    "pyrope_index_last_search_ms": (C.c_int, [vp, f32p]),
    "pyrope_index_last_search_launches": (C.c_int, [vp, i32p]),
    "pyrope_index_last_search_scanned": (C.c_int, [vp, i64p]),
    "pyrope_index_last_search_kernel": (C.c_int, [vp, f32p, C.POINTER(C.c_char_p)]),
    "pyrope_batcher_create": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(vp)]),
    "pyrope_batcher_create_sharded": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(vp)]),
    "pyrope_batcher_create_delta": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(vp)]),
    "pyrope_batcher_create_vindex": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(vp)]),
    "pyrope_batcher_destroy": (C.c_int, [vp]),
    "pyrope_batcher_search": (C.c_int, [vp, vp, C.c_int, C.c_int64, C.c_int, vp, vp, i32p]),
    "pyrope_batcher_stats": (C.c_int, [vp, i64p, i64p]),
    "pyrope_batcher_last_error": (C.c_char_p, []),
    "pyrope_topk_merge_device": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]),
    "pyrope_delta_create": (C.c_int, [vp, vp, C.POINTER(vp)]),
    "pyrope_delta_create_sharded": (C.c_int, [vp, vp, C.POINTER(vp)]),
    "pyrope_delta_destroy": (C.c_int, [vp]),
    "pyrope_delta_search_batch": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int64, C.c_int, vp, vp, vp]),
    "pyrope_delta_search_batch_topk": (C.c_int, [vp, C.c_int64, vp, vp, C.c_int64, C.c_int, vp, vp, vp]),
    "pyrope_delta_search_batch_device": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int64, C.c_int, vp, vp, vp, vp]),
    "pyrope_delta_compact": (C.c_int, [vp, i64p, vp]),
    "pyrope_delta_move": (C.c_int, [vp, i64p, vp]),
    "pyrope_delta_build_tail": (C.c_int, [vp]),
    "pyrope_delta_extend_tail": (C.c_int, [vp]),
    "pyrope_delta_stats": (C.c_int, [vp, i64p]),
    "pyrope_delta_snapshot": (C.c_int, [vp, C.c_char_p]),
    "pyrope_delta_load": (C.c_int, [vp, C.c_char_p]),
    "pyrope_vindex_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "pyrope_vindex_create_delta": (C.c_int, [vp, vp, C.POINTER(vp)]),
    "pyrope_vindex_create_sharded": (C.c_int, [C.c_int, i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "pyrope_vindex_destroy": (C.c_int, [vp]),
    "pyrope_vindex_native": (C.c_int, [vp, C.POINTER(vp)]),
    "pyrope_vindex_set_quantization": (C.c_int, [vp, C.c_int]),
    "pyrope_vindex_add": (C.c_int, [vp, C.c_char_p, vp, C.c_int]),
    "pyrope_vindex_upsert": (C.c_int, [vp, C.c_char_p, vp, C.c_int]),
    "pyrope_vindex_delete": (C.c_int, [vp, C.c_char_p, i32p]),
    "pyrope_vindex_build": (C.c_int, [vp]),
    "pyrope_vindex_extend": (C.c_int, [vp]),
    "pyrope_vindex_search": (C.c_int, [vp, C.c_int64, vp, C.c_int, C.c_int, C.c_int64, C.c_int, vp, vp, vp]),
    "pyrope_vindex_id": (C.c_int, [C.c_int64, C.c_char_p, C.c_int, i32p]),
    "pyrope_vindex_ids": (C.c_int, [vp, C.c_int64, vp, C.c_int64, vp, i64p]),
    "pyrope_vindex_id_table_size": (C.c_int, [i64p, i64p]),
    "pyrope_vindex_stats": (C.c_int, [vp, i64p, i32p, i32p]),
    "pyrope_vindex_get_centroids": (C.c_int, [vp, vp, i32p]),
    "pyrope_vindex_snapshot": (C.c_int, [vp, C.c_char_p]),
    "pyrope_vindex_load": (C.c_int, [vp, C.c_char_p]),
    "pyrope_vindex_last_error": (C.c_char_p, []),
    "pyrope_parse_vector": (C.c_int, [vp, C.c_int64, vp, C.c_int64, i64p]),
    "pyrope_encode_vector": (C.c_int, [vp, C.c_int64, vp, C.c_int64]),
    "pyrope_fvecs_read": (C.c_int, [C.c_char_p, C.c_int64, C.c_int64, vp, C.c_int64, i64p, i32p]),
    "pyrope_index_add_fvecs": (C.c_int, [vp, C.c_char_p, C.c_int64, i64p]),
    "pyrope_formats_last_error": (C.c_char_p, []),
    "pyrope_coarse_assign": (C.c_int, [C.c_int, C.c_int, C.c_int64, vp, C.c_int, vp, vp]),
    "pyrope_kmeans_train": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_int64, vp, C.c_int, C.c_int, C.c_int32, vp, i32p, i32p]),
    "pyrope_pq_encode": (C.c_int, [C.c_int, C.c_int, C.c_int, vp, vp, C.c_int64, vp, vp]),
    "pyrope_pq_distance_table": (C.c_int, [C.c_int, C.c_int, C.c_int, vp, C.c_int64, vp, vp]),
    "pyrope_fill_uniform_device": (C.c_int, [vp, C.c_int64, C.c_uint64, C.c_uint64, vp]),
}

_lib = None


def load():
    """Load the CUDA library.  Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PyropeGpuError(ERR_INVALID_STATE,
                             f"{LIB_PATH} is missing: build it with `python -m pyrope_b200.build` "
                             "(pyrope_b200 has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(code: int):
    if code != OK:
        msg = load().pyrope_last_error()
        raise PyropeGpuError(code, msg.decode("utf-8", "replace") if msg else "")


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _p(a):
    return a.ctypes.data_as(vp) if a is not None else None


class GpuIndex:
    """Thin, typed view of one pyrope_index handle (dense row ordinals, numpy in/out)."""

    def __init__(self, kind: int, dim: int, metric: int = L2, nlist: int = 100, m: int = 4, k: int = 256,
                 device: int | None = None):
        L = load()
        if device is not None:
            check(L.pyrope_gpu_init(device))
        h = vp()
        check(L.pyrope_index_create(kind, dim, metric, nlist, m, k, C.byref(h)))
        self._h = h
        self.kind, self.dim, self.metric, self.nlist, self.m, self.k = kind, dim, metric, nlist, m, k

    def close(self):
        if getattr(self, "_h", None):
            load().pyrope_index_destroy(self._h)
            self._h = None

    __del__ = close

    # ---- writes
    def reserve(self, n):
        check(load().pyrope_index_reserve(self._h, n))

    def add(self, X, labels=None) -> int:
        X = _np(X, np.float32)
        if X.ndim == 1:
            X = X[None, :]
        if X.shape[1] != self.dim:
            raise PyropeGpuError(ERR_DIMENSION, "Vector dimension mismatch")
        lab = _np(labels, np.int64) if labels is not None else None
        first = C.c_int64(-1)
        check(load().pyrope_index_add_batch(self._h, X.shape[0], _p(X), _p(lab), C.byref(first)))
        return first.value

    def add_device(self, ptr: int, n: int, labels_ptr: int | None = None) -> int:
        first = C.c_int64(-1)
        check(load().pyrope_index_add_batch_device(self._h, n, vp(ptr), vp(labels_ptr) if labels_ptr else None,
                                                   C.byref(first)))
        return first.value

    def update_row(self, row, x):
        x = _np(x, np.float32).reshape(-1)
        if x.size != self.dim:
            raise PyropeGpuError(ERR_DIMENSION, "Vector dimension mismatch")
        check(load().pyrope_index_update_row(self._h, row, _p(x)))

    def delete_row(self, row) -> bool:
        rc = load().pyrope_index_delete_row(self._h, row)
        if rc == ERR_NOT_FOUND:
            return False
        check(rc)
        return True

    def shadow_row(self, row, shadowed=True):
        check(load().pyrope_index_shadow_row(self._h, row, 1 if shadowed else 0))

    def set_quantization(self, enable: bool):
        check(load().pyrope_index_set_quantization(self._h, 1 if enable else 0))

    # ---- build
    def build(self):
        check(load().pyrope_index_build(self._h))

    def extend(self):
        """Append the write buffer to the built inverted lists without re-training (pyrope_index_extend)."""
        check(load().pyrope_index_extend(self._h))

    def set_train_params(self, max_train_rows=0, max_iter=0):
        check(load().pyrope_index_set_train_params(self._h, max_train_rows, max_iter))

    def set_codebooks(self, centroids, pq_codebooks=None):
        c = _np(centroids, np.float32)
        cb = _np(pq_codebooks, np.float32) if pq_codebooks is not None else None
        check(load().pyrope_index_set_codebooks(self._h, c.shape[0], _p(c), _p(cb)))

    def set_shard(self, rank, world):
        check(load().pyrope_index_set_shard(self._h, rank, world))

    def threshold_exchange_handle(self, max_queries: int) -> bytes:
        buf = C.create_string_buffer(64)
        check(load().pyrope_index_threshold_exchange_handle(self._h, max_queries, buf))
        return buf.raw

    def threshold_exchange_open(self, world: int, rank: int, handles: bytes):
        assert len(handles) == 64 * world
        check(load().pyrope_index_threshold_exchange_open(self._h, world, rank, handles))

    def threshold_exchange_close(self):
        check(load().pyrope_index_threshold_exchange_close(self._h))

    def threshold_exchange_epoch(self, epoch: int):
        check(load().pyrope_index_threshold_exchange_epoch(self._h, epoch))

    def is_built(self) -> bool:
        out = C.c_int32(0)
        check(load().pyrope_index_is_built(self._h, C.byref(out)))
        return bool(out.value)

    def centroids(self):
        n = C.c_int32(0)
        check(load().pyrope_index_get_centroids(self._h, None, C.byref(n)))
        if n.value == 0:
            return None
        out = np.zeros((n.value, self.dim), np.float32)
        check(load().pyrope_index_get_centroids(self._h, _p(out), C.byref(n)))
        return out

    def codebooks(self):
        cb = np.zeros((self.m, self.k, self.dim // self.m), np.float32)
        ks = np.zeros(self.m, np.int32)
        check(load().pyrope_index_get_codebooks(self._h, _p(cb), _p(ks)))
        return cb, ks

    def lists(self):
        """-> (offsets[nc+1], rows[total], codes[total][m] or None)"""
        tot = C.c_int64(0)
        check(load().pyrope_index_get_lists(self._h, None, None, None, C.byref(tot)))
        c = self.centroids()
        nc = 0 if c is None else c.shape[0]
        off = np.zeros(nc + 1, np.int64)
        rows = np.zeros(max(tot.value, 1), np.int64)
        codes = np.zeros((max(tot.value, 1), self.m), np.uint8) if self.kind == IVF_PQ else None
        check(load().pyrope_index_get_lists(self._h, _p(off), _p(rows), _p(codes), C.byref(tot)))
        return off, rows[:tot.value], (codes[:tot.value] if codes is not None else None)

    def snapshot(self, path: str):
        check(load().pyrope_index_snapshot(self._h, str(path).encode()))

    def load(self, path: str):
        check(load().pyrope_index_load(self._h, str(path).encode()))

    def stats(self):
        live, buf = C.c_int64(0), C.c_int64(0)
        dim, metric = C.c_int32(0), C.c_int32(0)
        check(load().pyrope_index_stats(self._h, C.byref(live), C.byref(buf), C.byref(dim), C.byref(metric)))
        return {"live": live.value, "buffer": buf.value, "dim": dim.value, "metric": metric.value}

    # ---- search
    def search(self, Q, topk: int, max_scans: int = -1, nprobe: int = -1):
        Q = _np(Q, np.float32)
        if Q.ndim == 1:
            Q = Q[None, :]
        if Q.shape[1] != self.dim:
            raise PyropeGpuError(ERR_DIMENSION, "Vector dimension mismatch")
        nq = Q.shape[0]
        kk = max(topk, 1)
        scores = np.zeros((nq, kk), np.float32)
        rows = np.full((nq, kk), -1, np.int64)
        counts = np.zeros(nq, np.int32)
        check(load().pyrope_index_search_batch(self._h, nq, _p(Q), topk, max_scans, nprobe, _p(scores), _p(rows),
                                               _p(counts)))
        return scores, rows, counts

    def search_device(self, q_ptr: int, nq: int, topk: int, scores_ptr: int, rows_ptr: int, counts_ptr: int,
                      max_scans: int = -1, nprobe: int = -1, stream: int | None = None):
        check(load().pyrope_index_search_batch_device(self._h, nq, vp(q_ptr), topk, max_scans, nprobe, vp(scores_ptr),
                                                      vp(rows_ptr), vp(counts_ptr), vp(stream) if stream else None))

    def coarse_probe_device(self, q_ptr: int, nq: int, nprobe: int, probes_ptr: int, stream: int | None = None):
        check(load().pyrope_index_coarse_probe_device(self._h, nq, vp(q_ptr), nprobe, vp(probes_ptr),
                                                      vp(stream) if stream else None))

    def search_probed_device(self, q_ptr: int, nq: int, topk: int, nprobe: int, probes_ptr: int, scores_ptr: int,
                             rows_ptr: int, counts_ptr: int, max_scans: int = -1, stream: int | None = None):
        check(load().pyrope_index_search_batch_probed_device(self._h, nq, vp(q_ptr), topk, max_scans, nprobe,
                                                             vp(probes_ptr), vp(scores_ptr), vp(rows_ptr),
                                                             vp(counts_ptr), vp(stream) if stream else None))

    def last_search_ms(self):
        out = (C.c_float * 4)()
        check(load().pyrope_index_last_search_ms(self._h, out))
        return {"total": out[0], "coarse": out[1], "scan": out[2], "merge": out[3]}

    def last_search_launches(self) -> int:
        out = C.c_int32(0)
        check(load().pyrope_index_last_search_launches(self._h, C.byref(out)))
        return out.value

    def last_search_kernel(self):
        """(name, ms) of the dominant kernel of the last search, timed alone with CUDA events."""
        ms = C.c_float(0)
        name = C.c_char_p()
        check(load().pyrope_index_last_search_kernel(self._h, C.byref(ms), C.byref(name)))
        return (name.value or b"").decode(), ms.value

    def last_search_scanned(self) -> int:
        """PQ codes scored by the last batched IVF_PQ search (sum of probed list lengths)."""
        out = C.c_int64(0)
        check(load().pyrope_index_last_search_scanned(self._h, C.byref(out)))
        return out.value


class _BorrowedIndex(GpuIndex):
    """Row-ordinal view of a handle somebody else owns (a shard of a ShardedIndex): never destroys it."""

    def close(self):
        self._h = None

    __del__ = close


class PeerGroup:
    """One rank's end of the all-gathers of a sharded search, over NVLink peer memory (pyrope_peer_*, csrc/peer.cu)."""

    def __init__(self, world: int, rank: int, slot_bytes: int, n_slots: int = 1):
        g = vp()
        self._g = None
        check(load().pyrope_peer_group_create(world, rank, slot_bytes, n_slots, C.byref(g)))
        self._g = g
        self.world, self.rank = world, rank

    def handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        check(load().pyrope_peer_group_handle(self._g, buf))
        return buf.raw

    def open(self, handles: bytes):
        assert len(handles) == 64 * self.world
        check(load().pyrope_peer_group_open(self._g, C.create_string_buffer(handles, len(handles))))

    def buffer(self) -> int:
        out = vp()
        check(load().pyrope_peer_group_buffer(self._g, C.byref(out)))
        return out.value

    def attach(self, buffers):
        arr = (vp * self.world)(*[vp(int(b)) if b else vp() for b in buffers])
        check(load().pyrope_peer_group_attach(self._g, arr))

    def allgather(self, slot: int, src_ptr: int, bytes_per_rank: int, stream: int = 0) -> int:
        """Enqueue the exchange on `stream`; returns the device address of [world][bytes_per_rank]."""
        out = vp()
        check(load().pyrope_peer_allgather_device(self._g, slot, vp(src_ptr), bytes_per_rank, C.byref(out), vp(stream)))
        return out.value

    def close(self):
        if getattr(self, "_g", None):
            load().pyrope_peer_group_destroy(self._g)
            self._g = None

    __del__ = close


class ShardedIndex:
    """One index over several GPUs of the box, driven by this one process (pyrope_sharded_*, csrc/sharded.cu)."""

    def __init__(self, n_devices: int, kind: int, dim: int, metric: int = L2, nlist: int = 100, m: int = 4, k: int = 256,
                 devices=None):
        s = vp()
        dv = _np(devices, np.int32) if devices is not None else None
        check(load().pyrope_sharded_create(n_devices, dv.ctypes.data_as(i32p) if dv is not None else None, kind, dim,
                                          metric, nlist, m, k, C.byref(s)))
        self._s, self.n, self.kind, self.dim, self.metric, self.nlist, self.m, self.k = s, n_devices, kind, dim, metric, nlist, m, k

    def close(self):
        if getattr(self, "_s", None):
            load().pyrope_sharded_destroy(self._s)
            self._s = None

    __del__ = close

    def shard(self, i: int):
        """(borrowed GpuIndex view of shard i, its CUDA device ordinal)"""
        h, dev = vp(), C.c_int32(0)
        check(load().pyrope_sharded_shard(self._s, i, C.byref(h), C.byref(dev)))
        g = _BorrowedIndex.__new__(_BorrowedIndex)
        g._h, g.kind, g.dim, g.metric, g.nlist, g.m, g.k = h, self.kind, self.dim, self.metric, self.nlist, self.m, self.k
        g._owner = self  # keep the sharded object alive while the view is in use
        return g, dev.value

    def note_rows(self, total: int):
        check(load().pyrope_sharded_note_rows(self._s, total))

    def set_train_params(self, max_train_rows=0, max_iter=0):
        check(load().pyrope_sharded_set_train_params(self._s, max_train_rows, max_iter))

    def set_codebooks(self, centroids, pq_codebooks=None):
        c = _np(centroids, np.float32)
        cb = _np(pq_codebooks, np.float32) if pq_codebooks is not None else None
        check(load().pyrope_sharded_set_codebooks(self._s, c.shape[0], _p(c), _p(cb)))

    def add(self, X, labels=None) -> int:
        X = _np(X, np.float32)
        if X.ndim == 1:
            X = X[None, :]
        if X.shape[1] != self.dim:
            raise PyropeGpuError(ERR_DIMENSION, "Vector dimension mismatch")
        lab = _np(labels, np.int64) if labels is not None else None
        first = C.c_int64(-1)
        check(load().pyrope_sharded_add_batch(self._s, X.shape[0], _p(X), _p(lab), C.byref(first)))
        return first.value

    def delete_row(self, row: int) -> bool:
        rc = load().pyrope_sharded_delete_row(self._s, row)
        if rc == ERR_NOT_FOUND:
            return False
        check(rc)
        return True

    def update_row(self, row: int, x):
        x = _np(x, np.float32).reshape(-1)
        if x.size != self.dim:
            raise PyropeGpuError(ERR_DIMENSION, "Vector dimension mismatch")
        check(load().pyrope_sharded_update_row(self._s, row, _p(x)))

    def shadow_row(self, row: int, shadowed=True):
        check(load().pyrope_sharded_shadow_row(self._s, row, 1 if shadowed else 0))

    def set_labels(self, labels_by_row):
        lab = _np(labels_by_row, np.int64)
        check(load().pyrope_sharded_set_labels(self._s, lab.size, _p(lab)))

    def build(self):
        check(load().pyrope_sharded_build(self._s))

    def extend(self):
        """pyrope_sharded_extend: every shard appends the buffer to the lists it owns, all or nothing."""
        check(load().pyrope_sharded_extend(self._s))

    def is_built(self) -> bool:
        out = C.c_int32(0)
        check(load().pyrope_sharded_is_built(self._s, C.byref(out)))
        return bool(out.value)

    def centroids(self):
        n = C.c_int32(0)
        check(load().pyrope_sharded_get_centroids(self._s, None, C.byref(n)))
        if n.value == 0:
            return None
        out = np.zeros((n.value, self.dim), np.float32)
        check(load().pyrope_sharded_get_centroids(self._s, _p(out), C.byref(n)))
        return out

    def codebooks(self):
        cb = np.zeros((self.m, self.k, self.dim // self.m), np.float32)
        ks = np.zeros(self.m, np.int32)
        check(load().pyrope_sharded_get_codebooks(self._s, _p(cb), _p(ks)))
        return cb, ks

    def snapshot(self, path: str):
        check(load().pyrope_sharded_snapshot(self._s, str(path).encode()))

    def load(self, path: str):
        check(load().pyrope_sharded_load(self._s, str(path).encode()))

    def stats(self) -> int:
        out = C.c_int64(0)
        check(load().pyrope_sharded_stats(self._s, C.byref(out)))
        return out.value

    def search(self, Q, topk: int, max_scans: int = -1, nprobe: int = -1):
        Q = _np(Q, np.float32)
        if Q.ndim == 1:
            Q = Q[None, :]
        nq, kk = Q.shape[0], max(topk, 1)
        scores, rows, counts = np.zeros((nq, kk), np.float32), np.full((nq, kk), -1, np.int64), np.zeros(nq, np.int32)
        check(load().pyrope_sharded_search_batch(self._s, nq, _p(Q), topk, max_scans, nprobe, _p(scores), _p(rows), _p(counts)))
        return scores, rows, counts

    def search_device(self, q_ptr: int, nq: int, topk: int, scores_ptr: int, rows_ptr: int, counts_ptr: int, nprobe: int = -1):
        check(load().pyrope_sharded_search_batch_device(self._s, nq, vp(q_ptr), topk, -1, nprobe, vp(scores_ptr), vp(rows_ptr),
                                                       vp(counts_ptr)))

    def last_search_ms(self) -> float:
        out = C.c_float(0)
        check(load().pyrope_sharded_last_search_ms(self._s, C.byref(out)))
        return out.value


class Batcher:
    """Host micro-batcher (csrc/batcher.cu): search() blocks like IVectorIndex.Search does; concurrent callers
    share one batched launch.  ctypes drops the GIL during the call, so Python threads batch for real.

    target: a GpuIndex (rows = row ordinals / labels), a ShardedIndex (global row ordinals), a raw pyrope_delta handle
    (labels) or any vector_index object (id ordinals; vector_index.VectorIndexBatcher turns them into strings).  The
    batcher borrows the target and keeps a reference to it."""

    def __init__(self, target, max_batch: int = 256, max_wait_us: int = 200):
        L, b = load(), vp()
        if isinstance(target, GpuIndex):
            rc = L.pyrope_batcher_create(target._h, max_batch, max_wait_us, C.byref(b))
        elif isinstance(target, ShardedIndex):
            rc = L.pyrope_batcher_create_sharded(target._s, max_batch, max_wait_us, C.byref(b))
        elif hasattr(target, "_v"):  # a vector_index object (string ids)
            rc = L.pyrope_batcher_create_vindex(target._v, max_batch, max_wait_us, C.byref(b))
        elif isinstance(target, (vp, int)):  # a pyrope_delta handle
            rc = L.pyrope_batcher_create_delta(target, max_batch, max_wait_us, C.byref(b))
        else:
            raise TypeError(f"cannot batch searches of {type(target).__name__}")
        check(rc)
        self._b, self._index = b, target

    def search(self, q, topk: int, max_scans: int = -1, nprobe: int = -1):
        q = _np(q, np.float32).reshape(-1)
        kk = max(topk, 1)
        scores, rows, cnt = np.zeros(kk, np.float32), np.full(kk, -1, np.int64), C.c_int32(0)
        check(load().pyrope_batcher_search(self._b, _p(q), topk, max_scans, nprobe, _p(scores), _p(rows), C.byref(cnt)))
        return scores[:cnt.value], rows[:cnt.value]

    def stats(self):
        a, b = C.c_int64(0), C.c_int64(0)
        check(load().pyrope_batcher_stats(self._b, C.byref(a), C.byref(b)))
        return {"batches": a.value, "queries": b.value}

    def close(self):
        if getattr(self, "_b", None):
            load().pyrope_batcher_destroy(self._b)
            self._b = None

    __del__ = close


# ---- building blocks ---------------------------------------------------------------------------
def coarse_assign(X, centroids, metric=L2):
    X = _np(X, np.float32)
    c = _np(centroids, np.float32)
    out = np.zeros(X.shape[0], np.int32)
    check(load().pyrope_coarse_assign(metric, X.shape[1], X.shape[0], _p(X), c.shape[0], _p(c), _p(out)))
    return out


def kmeans_train(data, k, metric=L2, max_iter=10, seed=42):
    d = _np(data, np.float32)
    n, dim = d.shape
    kk = max(1, min(k if k > 0 else 1, n))
    out = np.zeros((kk, dim), np.float32)
    ko, it = C.c_int32(0), C.c_int32(0)
    check(load().pyrope_kmeans_train(metric, dim, n, dim, _p(d), k, max_iter, seed, _p(out), C.byref(ko), C.byref(it)))
    return out[:ko.value], it.value


def pq_encode(codebooks, X, ksub=None):
    cb = _np(codebooks, np.float32)
    m, k, sub = cb.shape
    X = _np(X, np.float32)
    ks = _np(ksub, np.int32) if ksub is not None else None
    out = np.zeros((X.shape[0], m), np.uint8)
    check(load().pyrope_pq_encode(m * sub, m, k, _p(cb), _p(ks), X.shape[0], _p(X), _p(out)))
    return out


def pq_distance_table(codebooks, Q):
    cb = _np(codebooks, np.float32)
    m, k, sub = cb.shape
    Q = _np(Q, np.float32)
    out = np.zeros((Q.shape[0], m, k), np.float32)
    check(load().pyrope_pq_distance_table(m * sub, m, k, _p(cb), Q.shape[0], _p(Q), _p(out)))
    return out


def topk_merge_device(nq, parts, k_in, k_out, scores_ptr, rows_ptr, out_scores_ptr, out_rows_ptr, out_counts_ptr,
                      stream=None):
    check(load().pyrope_topk_merge_device(nq, parts, k_in, k_out, vp(scores_ptr), vp(rows_ptr), vp(out_scores_ptr),
                                          vp(out_rows_ptr), vp(out_counts_ptr) if out_counts_ptr else None,
                                          vp(stream) if stream else None))


def fill_uniform_device(ptr, n, seed, offset=0, stream=None):
    check(load().pyrope_fill_uniform_device(vp(ptr), n, seed, offset, vp(stream) if stream else None))
