"""GPU parity of the query-stationary tensor-core coarse probe (csrc/coarse_tc.cu): the probed lists — and hence the
search results — must equal the oracle's ranking of ALL centroids in the reference's arithmetic
(IvfFlatVectorIndex.cs:186-198, IvfPqVectorIndex.cs:141-150), for every metric, for tables that take whole-unit maxima
(>= 2 k' units of 128 centroids) and 32-column maxima (smaller tables), with ragged sizes, and when thousands of
centroids crowd one rounding band (duplicates: the exhaustive fallback)."""
import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.parity import assert_batch_equivalent
from tests.test_gpu_flat_tc_regimes import in_child  # noqa: F401  (fixture: runs a function in a child process)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    import pyrope_b200 as pg
    pg._lib.check(pg.load().pyrope_gpu_init(0))
    return pg


def _frozen_pair(gpu, metric, dim, nlist, n, seed, dup=0):
    """IVF_PQ index over n random rows with GIVEN codebooks (random centroids, random PQ codewords): the build only
    assigns and encodes, the oracle adopts the result, so a search compares the coarse ranking + scan alone."""
    rng = np.random.default_rng(seed)
    cent = rng.random((nlist, dim), dtype=np.float32)
    if dup:                                      # a crowd of near-identical centroids (distinct in fp32, one TF32 band)
        cent[100:100 + dup] = cent[7] + (rng.random((dup, dim), dtype=np.float32) - 0.5) * 2e-3
    cb = (rng.random((16, 256, dim // 16), dtype=np.float32) - 0.5) * 0.5
    base = rng.random((n, dim), dtype=np.float32)
    gm = {"L2": gpu.L2, "IP": gpu.INNER_PRODUCT, "COSINE": gpu.COSINE}[metric]
    om = {"L2": orc.L2, "IP": orc.IP, "COSINE": orc.COSINE}[metric]
    ix = gpu.GpuIndex(gpu.IVF_PQ, dim, gm, nlist=nlist, m=16, k=256)
    ix.set_codebooks(cent, cb)
    ix.add(base)
    ix.build()
    off, rows, codes = ix.lists()
    ref = orc.IvfPqIndex(dim, om, m=16, k=256, nlist=nlist)
    ref.adopt(cent, cb, off, rows, codes)
    return ix, ref, rng


def _s(ix, Q, k, **kw):
    sc, rows, cnt = ix.search(Q, k, **kw)
    return rows, sc, cnt


@pytest.mark.parametrize("metric,dim,nlist,nprobe", [
    ("L2", 128, 40000, 64),     # whole-unit maxima (313 units >= 2 x 72)
    ("L2", 128, 9001, 32),      # 32-column maxima, ragged last unit
    ("IP", 128, 20000, 16),
    ("COSINE", 64, 12000, 8),   # dim 64: two K chunks, per-centroid scale
    ("L2", 32, 2500, 4),        # smallest table the path takes
])
def test_coarse_probe_matches_oracle(gpu, metric, dim, nlist, nprobe):
    ix, ref, rng = _frozen_pair(gpu, metric, dim, nlist, 120_000, seed=nlist)
    for nq in (700, 3):         # several resident query tiles / a ragged single tile
        Q = rng.random((nq, dim), dtype=np.float32)
        assert_batch_equivalent(ref.search_batch(Q, 10, nprobe=nprobe), _s(ix, Q, 10, nprobe=nprobe),
                                ctx=f"coarse {metric} d={dim} nlist={nlist} nprobe={nprobe} nq={nq}")


def test_coarse_probe_with_a_crowd_of_duplicate_centroids(gpu):
    """3,000 near-identical centroids sit inside one rounding band: queries near them overflow the candidate list and
    are ranked exhaustively; the result must still be the oracle's."""
    ix, ref, rng = _frozen_pair(gpu, "L2", 128, 20000, 60_000, seed=5, dup=3000)
    cent7 = ix.centroids()[7]
    Q = rng.random((64, 128), dtype=np.float32)
    Q[:16] = cent7 + (rng.random((16, 128), dtype=np.float32) - 0.5) * 1e-3   # right on top of the crowd
    assert_batch_equivalent(ref.search_batch(Q, 10, nprobe=32), _s(ix, Q, 10, nprobe=32), ctx="duplicate centroids")


def test_coarse_probe_agrees_with_streaming_kernel(gpu, monkeypatch):
    ix, ref, rng = _frozen_pair(gpu, "L2", 128, 30000, 80_000, seed=11)
    Q = rng.random((300, 128), dtype=np.float32)
    a = _s(ix, Q, 10, nprobe=24)
    monkeypatch.setenv("PYROPE_COARSE_STREAMING", "1")
    b = _s(ix, Q, 10, nprobe=24)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)


# ------------------------------------------------------------------------------------------------
# the tensor passes run on fp16 copies (L2 / IP): values outside what fp16 holds must not cost exactness
# ------------------------------------------------------------------------------------------------
def _frozen_from(gpu, metric, cent, base, seed=0):
    dim, nlist = cent.shape[1], cent.shape[0]
    rng = np.random.default_rng(seed)
    spread = float(np.abs(base).mean()) or 1.0
    cb = ((rng.random((16, 256, dim // 16), dtype=np.float32) - 0.5) * np.float32(0.5 * spread)).astype(np.float32)
    gm = {"L2": gpu.L2, "IP": gpu.INNER_PRODUCT}[metric]
    om = {"L2": orc.L2, "IP": orc.IP}[metric]
    ix = gpu.GpuIndex(gpu.IVF_PQ, dim, gm, nlist=nlist, m=16, k=256)
    ix.set_codebooks(cent, cb)
    ix.add(base)
    ix.build()
    off, rows, codes = ix.lists()
    ref = orc.IvfPqIndex(dim, om, m=16, k=256, nlist=nlist)
    ref.adopt(cent, cb, off, rows, codes)
    return ix, ref


@pytest.mark.parametrize("metric", ["L2", "IP"])
def test_coarse_probe_tiny_values_underflow_fp16(gpu, metric):
    """Every value below fp16's smallest normal (6.1e-5): the copies hold subnormals and zeros, the bound must carry their
    absolute error."""
    rng = np.random.default_rng(41)
    cent = (rng.random((6000, 128), dtype=np.float32) * np.float32(3e-5)).astype(np.float32)
    base = (rng.random((40_000, 128), dtype=np.float32) * np.float32(3e-5)).astype(np.float32)
    ix, ref = _frozen_from(gpu, metric, cent, base)
    Q = (rng.random((300, 128), dtype=np.float32) * np.float32(3e-5)).astype(np.float32)
    assert_batch_equivalent(ref.search_batch(Q, 10, nprobe=16), _s(ix, Q, 10, nprobe=16), ctx=f"tiny values {metric}")


def test_coarse_probe_mixed_magnitudes(gpu):
    """Dimensions eight orders of magnitude apart inside one row: large ones near the top of the fp16 range, small ones
    underflowing."""
    rng = np.random.default_rng(42)
    mag = np.where(np.arange(128) % 4 == 0, np.float32(2.0e4), np.float32(1e-4)).astype(np.float32)
    cent = (rng.random((5000, 128), dtype=np.float32) * mag).astype(np.float32)
    base = (rng.random((30_000, 128), dtype=np.float32) * mag).astype(np.float32)
    ix, ref = _frozen_from(gpu, "L2", cent, base)
    Q = (rng.random((200, 128), dtype=np.float32) * mag).astype(np.float32)
    assert_batch_equivalent(ref.search_batch(Q, 10, nprobe=16), _s(ix, Q, 10, nprobe=16), ctx="mixed magnitudes")


def test_coarse_probe_values_beyond_fp16(gpu):
    """A query with a component fp16 cannot hold is ranked exhaustively; a centroid table with one keeps the tf32 passes."""
    rng = np.random.default_rng(43)
    cent = rng.random((6000, 128), dtype=np.float32)
    base = rng.random((40_000, 128), dtype=np.float32)
    ix, ref = _frozen_from(gpu, "L2", cent, base)
    Q = rng.random((260, 128), dtype=np.float32)
    Q[5, 17] = np.float32(1.0e5)
    Q[258, 0] = np.float32(-7.0e4)
    assert_batch_equivalent(ref.search_batch(Q, 10, nprobe=16), _s(ix, Q, 10, nprobe=16), ctx="query beyond fp16")
    cent2 = cent.copy()
    cent2[1234, 5] = np.float32(9.0e4)
    ix2, ref2 = _frozen_from(gpu, "L2", cent2, base)
    Q2 = rng.random((100, 128), dtype=np.float32)
    assert_batch_equivalent(ref2.search_batch(Q2, 10, nprobe=16), _s(ix2, Q2, 10, nprobe=16), ctx="centroid beyond fp16")


def _coarse_pass_case(gpu):
    rng = np.random.default_rng(44)
    cent = rng.random((30000, 128), dtype=np.float32)
    base = rng.random((80_000, 128), dtype=np.float32)
    ix, ref = _frozen_from(gpu, "L2", cent, base)
    Q = rng.random((300, 128), dtype=np.float32)
    return ix, ref, Q


def _cold_warm(ix, Q):
    """Search twice: (result, launches of the first search, launches of the second)."""
    a = _s(ix, Q, 10, nprobe=24)
    cold = ix.last_search_launches()
    b = _s(ix, Q, 10, nprobe=24)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    return a, cold, ix.last_search_launches()


def child_coarse_passes(out):
    """Child-process side of the test below (PYROPE_COARSE_TF32 is read once per process)."""
    import pyrope_b200 as pg
    pg._lib.check(pg.load().pyrope_gpu_init(0))
    ix, _, Q = _coarse_pass_case(pg)
    (rows, sc, cnt), cold, warm = _cold_warm(ix, Q)
    np.savez(out, rows=rows, scores=sc, counts=cnt, cold=cold, warm=warm)


def test_coarse_probe_fp16_and_tf32_passes_agree(gpu, in_child):
    """The same frozen IVF_PQ index probed by the fp16 passes (default) and, in a child process, by the tf32 passes
    (PYROPE_COARSE_TF32=1): identical results, both the oracle's.  Only the fp16 passes convert the centroid table, on the
    first search."""
    ix, ref, Q = _coarse_pass_case(gpu)
    a, cold, warm = _cold_warm(ix, Q)
    assert_batch_equivalent(ref.search_batch(Q, 10, nprobe=24), a, ctx="fp16 passes")
    b = in_child({"PYROPE_COARSE_TF32": "1"}, "tests.test_gpu_coarse:child_coarse_passes")
    for x, y in zip(a, (b["rows"], b["scores"], b["counts"])):
        np.testing.assert_array_equal(x, y)
    assert cold - warm == int(b["cold"]) - int(b["warm"]) + 1, (cold, warm, int(b["cold"]), int(b["warm"]))
