"""The library keeps one thread-local error message: whichever module raised the error, pyrope_last_error() and every
per-module reader kept for existing shims return the same bytes.  Every failure below is an argument check made before
any CUDA call, so this runs without a GPU."""
import ctypes as C
import threading

import pytest

from pyrope_b200 import _lib

READERS = ("pyrope_last_error", "pyrope_sharded_last_error", "pyrope_peer_last_error", "pyrope_batcher_last_error",
           "pyrope_vindex_last_error", "pyrope_formats_last_error")
MISSING = b"/nonexistent/pyrope-error-channel.fvecs"

# module -> (a failing call, its status, its message)
CASES = {
    "sharded": (lambda L: L.pyrope_sharded_add_batch(None, 1, None, None, None), _lib.ERR_INVALID_ARG, b"handle is null"),
    "vindex": (lambda L: L.pyrope_vindex_add(None, b"a", None, 4), _lib.ERR_INVALID_ARG, b"index handle is null"),
    "batcher": (lambda L: L.pyrope_batcher_search(None, None, 10, -1, -1, None, None, None), _lib.ERR_INVALID_ARG,
                b"null argument"),
    "peer": (lambda L: L.pyrope_peer_group_create(0, 0, 64, 1, C.byref(C.c_void_p())), _lib.ERR_INVALID_ARG,
             b"world must be 2..8, rank below it"),
    "formats": (lambda L: L.pyrope_fvecs_read(MISSING, -1, 0, None, 0, None, None), _lib.ERR_NOT_FOUND,
                b"Could not find file '" + MISSING + b"'."),
    "index_add_fvecs": (lambda L: L.pyrope_index_add_fvecs(None, MISSING, -1, C.byref(C.c_int64())), _lib.ERR_INVALID_ARG,
                        b"index handle is null"),
}


def _messages(L):
    return [getattr(L, r)() for r in READERS]


@pytest.mark.parametrize("module", list(CASES))
def test_every_reader_returns_the_failing_call_message(module):
    L = _lib.load()
    call, status, message = CASES[module]
    # a different message first: the call under test must replace it, not find its own text there
    assert L.pyrope_fvecs_read(None, -1, 0, None, 0, None, None) == _lib.ERR_INVALID_ARG
    assert L.pyrope_last_error() == b"Value cannot be null. (Parameter 'path')"
    assert call(L) == status
    assert _messages(L) == [message] * len(READERS)


def test_a_failure_on_another_thread_leaves_this_thread_message():
    L = _lib.load()
    sharded, _, sharded_msg = CASES["sharded"]
    peer, _, peer_msg = CASES["peer"]
    assert sharded(L) != _lib.OK
    seen = []
    t = threading.Thread(target=lambda: seen.append((peer(L), _messages(L))))
    t.start()
    t.join()
    assert seen == [(_lib.ERR_INVALID_ARG, [peer_msg] * len(READERS))]
    assert _messages(L) == [sharded_msg] * len(READERS)
