"""Payload and dataset formats either side of the scan path, by the reference's names (ctypes -> csrc/formats.cu):
VectorParsing.ParseVector (Utils/VectorParsing.cs), VectorEncoding.ToLittleEndianBytes
(Benchmarks/Encoding/VectorEncoding.cs), FvecsReader.Read (Benchmarks/Datasets/FvecsReader.cs)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import _p, vp


class FormatException(ValueError):
    pass


def _err():
    return (_lib.load().pyrope_last_error() or b"").decode("utf-8", "replace")


def _ck(rc):
    if rc == _lib.OK:
        return
    msg = _err()
    if rc == _lib.ERR_NOT_FOUND:
        raise FileNotFoundError(msg)
    if "Unsupported vector format" in msg or "out of bounds" in msg:
        raise FormatException(msg)
    if "Truncated" in msg:
        raise EOFError(msg)
    raise ValueError(msg)


def ParseVector(data: bytes) -> np.ndarray:
    data = bytes(data)
    n = C.c_int64(0)
    buf = (C.c_uint8 * max(len(data), 1)).from_buffer_copy(data or b"\0")
    _ck(_lib.load().pyrope_parse_vector(buf if data else None, len(data), None, 0, C.byref(n)))
    out = np.zeros(n.value, np.float32)
    _ck(_lib.load().pyrope_parse_vector(buf, len(data), _p(out), n.value, C.byref(n)))
    return out


def ToLittleEndianBytes(vector) -> bytes:
    if vector is None:
        raise ValueError("Value cannot be null. (Parameter 'vector')")
    v = np.ascontiguousarray(vector, np.float32).reshape(-1)
    out = (C.c_uint8 * max(v.size * 4, 1))()
    _ck(_lib.load().pyrope_encode_vector(_p(v), v.size, out, v.size * 4))
    return bytes(out)[:v.size * 4]


def ReadFvecs(path: str, limit: int | None = None, skip: int = 0) -> np.ndarray:
    """-> [count][dim] float32 (FvecsReader.Read yields the same rows one by one)."""
    if path is None:
        raise ValueError("Value cannot be null. (Parameter 'path')")
    lim = -1 if limit is None else (0 if limit <= 0 else int(limit))
    cnt, dim = C.c_int64(0), C.c_int32(0)
    _ck(_lib.load().pyrope_fvecs_read(str(path).encode(), lim, skip, None, 0, C.byref(cnt), C.byref(dim)))
    out = np.zeros((cnt.value, max(dim.value, 0)), np.float32)
    if cnt.value:
        _ck(_lib.load().pyrope_fvecs_read(str(path).encode(), lim, skip, _p(out), out.size, C.byref(cnt), C.byref(dim)))
    return out


def AddFvecs(index: _lib.GpuIndex, path: str, limit: int | None = None) -> int:
    """Stream an fvecs file into a GPU index (64 MiB batches); returns the rows added."""
    lim = -1 if limit is None else (0 if limit <= 0 else int(limit))
    added = C.c_int64(0)
    _ck(_lib.load().pyrope_index_add_fvecs(index._h, str(path).encode(), lim, C.byref(added)))
    return added.value
