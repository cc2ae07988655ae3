"""The FLAT tensor-core scan (flat_tc.cu) in every regime run_tc / launch_flat_tc_select dispatch to, checked twice:

- against the oracle (tests/parity.py: ids equal modulo ties, scores within 1e-4, bit-identical where the ids agree);
- against a float64 reference of the same scan (f64_check): every returned score is its row's float64 score, and no
  scanned live row left out scores above the k-th returned one.  This catches a row the kernel drops even when the
  oracle's list and the GPU's are tie-equivalent.

Regimes (default PYROPE_FLAT_TC: tensor cores from 8,192 scanned rows; k' = k + (16 if k < 64 else 32), k' <= 224):

  3xTF32, one pass     d <= 256 and (n_scan < 16,384 or k' < 32); d > 256 and n_scan < 65,536
  two-pass             d <= 256, n_scan >= 16,384, k' >= 32               (3xTF32 name, >= 7 launches)
  1xFP16 + band        d > 256, n_scan >= 65,536, L2 / IP, d % 8 == 0, every table value within fp16's range
  1xTF32 + band        the same, but cosine, d % 8 != 0 or a table value beyond fp16

Process-wide switches read once per process (PYROPE_FLAT_TF32, _NOCLUSTER, _CLUSTER, PYROPE_COARSE_TF32) are run in a
child process that writes its results to an .npz; the per-search ones (PYROPE_TC_3X, _PASSA_3X, _PASSB_3X) in-process."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.parity import assert_batch_equivalent

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NT = orc.max_threads()
EPS32 = 2.0 ** -23

K3X, KF16, KTF32 = "flat_tc_kernel (3xTF32)", "flat_tc_kernel (1xFP16 + band)", "flat_tc_kernel (1xTF32 + band)"
METRICS = {"L2": orc.L2, "IP": orc.IP, "COSINE": orc.COSINE}


# ------------------------------------------------------------------------------------------------
# float64 reference
# ------------------------------------------------------------------------------------------------
def _fp32_norms(X):
    """Row norms in the reference's fp32 order (orc.norm): the cosine zero-or-not decision is taken on these."""
    return np.array([orc.norm(x) for x in X], dtype=np.float32)


def f64_scores(base, Q, metric, xnorm32=None):
    """[nq][n] float64 scores: -|q-x|^2, q.x, or q.x / (|q||x|) (0 where the reference's fp32 norm is below 1e-6)."""
    X = np.asarray(base, np.float64)
    Qd = np.asarray(Q, np.float64)
    dots = Qd @ X.T
    if metric == orc.L2:
        return -((Qd * Qd).sum(1)[:, None] + (X * X).sum(1)[None, :] - 2.0 * dots)
    if metric == orc.IP:
        return dots
    xn32 = _fp32_norms(base) if xnorm32 is None else xnorm32
    qn32 = _fp32_norms(Q)
    s = dots / (np.sqrt((Qd * Qd).sum(1))[:, None] * np.sqrt((X * X).sum(1))[None, :] + 1e-300)
    s[qn32 < 1e-6, :] = 0.0
    s[:, xn32 < 1e-6] = 0.0
    return s


def f64_check(base, live_mask, scanned_upto, Q, metric, got, S=None, ctx=""):
    """got = (rows [nq][k], scores [nq][k], counts [nq]) of a search over rows [0, scanned_upto) of `base` whose
    live_mask is set.  Tolerance: 1e-4 |s| plus the fp32 summation bound 4 ulp x d x (|q| max|x|) (|q| + max|x|)^2 for
    L2, 1 for cosine), so scores near 0 do not trip it.  S: precomputed f64_scores(base, Q, metric)."""
    base = np.asarray(base, np.float32)
    n, d = base.shape
    rows, sc, cnt = got
    k = rows.shape[1]
    scanned = np.zeros(n, bool)
    scanned[:scanned_upto] = True
    scanned &= np.asarray(live_mask, bool)
    S = f64_scores(base, Q, metric) if S is None else S
    Q64 = np.asarray(Q, np.float64)
    xmax = float(np.sqrt((base[scanned].astype(np.float64) ** 2).sum(1)).max()) if scanned.any() else 0.0
    n_live = int(scanned.sum())
    for q in range(len(cnt)):
        qn = float(np.sqrt((Q64[q] ** 2).sum()))
        scale = (qn + xmax) ** 2 if metric == orc.L2 else (qn * xmax if metric == orc.IP else 1.0)
        atol = 4.0 * EPS32 * d * scale

        def tol(s):
            return 1e-4 * abs(s) + atol

        c = int(cnt[q])
        assert c == min(k, n_live), f"{ctx} q{q}: count {c}, expected min({k}, {n_live})"
        r = np.asarray(rows[q][:c], np.int64)
        assert len(set(r.tolist())) == c, f"{ctx} q{q}: duplicate rows"
        assert (r >= 0).all() and (r < n).all() and scanned[r].all(), f"{ctx} q{q}: a returned row was not scanned live"
        for i in range(c):
            want = S[q, r[i]]
            assert abs(float(sc[q][i]) - want) <= tol(want), \
                f"{ctx} q{q}: row {r[i]} at rank {i} scored {float(sc[q][i])!r}, float64 {want!r}"
        if c == 0:
            continue
        rest = scanned.copy()
        rest[r] = False
        if rest.any():
            s_rest = np.where(rest, S[q], -np.inf)
            j = int(np.argmax(s_rest))
            kth = float(sc[q][c - 1])
            assert s_rest[j] <= kth + tol(kth), \
                f"{ctx} q{q}: missing row {j} scores {s_rest[j]!r} in float64, above the k-th returned {kth!r}"


def test_f64_check_accepts_oracle_and_rejects_a_dropped_row():
    """CPU: the reference check agrees with the oracle on all three metrics, and flags a result with its best row
    removed (the (k+1)-th row moved up in its place)."""
    rng = np.random.default_rng(9)
    base = (rng.random((400, 24), dtype=np.float32) - 0.3).astype(np.float32)
    base[7] = 0.0                                                          # a zero row: cosine scores it 0
    Q = (rng.random((12, 24), dtype=np.float32) - 0.3).astype(np.float32)
    live = np.ones(400, bool)
    live[rng.choice(400, 40, replace=False)] = False
    for name, metric in METRICS.items():
        ref = orc.FlatIndex(24, metric)
        ref.add_batch(base)
        for r in np.flatnonzero(~live):
            assert ref.delete(int(r))
        for ms, upto in ((-1, 400), (150, int(np.flatnonzero(live)[149]) + 1)):
            got = ref.search_batch(Q, 10, max_scans=ms, nthreads=NT)
            f64_check(base, live, upto, Q, metric, got, ctx=f"oracle {name} ms={ms}")
        rid, rsc, rcn = ref.search_batch(Q, 11, nthreads=NT)
        bad = (rid[:, 1:].copy(), rsc[:, 1:].copy(), np.minimum(rcn, 10))
        with pytest.raises(AssertionError, match="missing row"):
            f64_check(base, live, 400, Q, metric, bad, ctx=f"dropped {name}")


# ------------------------------------------------------------------------------------------------
# GPU fixtures and helpers
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    import pyrope_b200 as pg
    pg._lib.check(pg.load().pyrope_gpu_init(0))
    return pg


def _gm(pg, metric):
    return {orc.L2: pg.L2, orc.IP: pg.INNER_PRODUCT, orc.COSINE: pg.COSINE}[metric]


def _s(ix, Q, k, **kw):
    sc, rows, cnt = ix.search(Q, k, **kw)
    return rows, sc, cnt


def _data(n, d, seed):
    """Seeded table: standard normal rows (both signs, IP scores near 0 occur)."""
    return np.random.default_rng(seed).standard_normal((n, d), dtype=np.float32)


def _queries(nq, d, seed):
    return np.random.default_rng(seed + 1_000_003).standard_normal((nq, d), dtype=np.float32)


class Pair:
    """A GPU FLAT index next to the oracle's and the row table both hold (row ordinal = oracle id)."""

    def __init__(self, pg, metric, base, kind=None):
        self.pg, self.metric = pg, metric
        self.base = np.array(base, np.float32)
        self.live = np.ones(len(base), bool)
        d = base.shape[1]
        if kind is None or kind == pg.FLAT:
            self.ref = orc.FlatIndex(d, metric)
            self.ix = pg.GpuIndex(pg.FLAT, d, _gm(pg, metric))
        else:
            self.ref = orc.IvfFlatIndex(d, metric, nlist=64)
            self.ix = pg.GpuIndex(kind, d, _gm(pg, metric), nlist=64)
        self.ref.add_batch(self.base)
        self.ix.add(self.base)
        self._xn = None

    def append(self, X):
        X = np.asarray(X, np.float32).reshape(-1, self.base.shape[1])
        n0 = len(self.base)
        self.ref.add_batch(X, ids=np.arange(n0, n0 + len(X)))
        assert self.ix.add(X) == n0
        self.base = np.concatenate([self.base, X])
        self.live = np.concatenate([self.live, np.ones(len(X), bool)])
        self._xn = None

    def update(self, row, v):
        v = np.asarray(v, np.float32)
        self.ref.upsert(int(row), v)
        self.ix.update_row(int(row), v)
        self.base[row] = v
        self.live[row] = True
        self._xn = None

    def delete(self, row):
        assert self.ref.delete(int(row)) and self.ix.delete_row(int(row))
        self.live[row] = False

    def cutoff(self, max_scans):
        """segment_cutoff: the scan position at which exactly min(max_scans, live) live rows precede it."""
        if max_scans < 0:
            return len(self.base)
        pos = np.flatnonzero(self.live)
        return int(pos[max_scans - 1]) + 1 if 0 < max_scans <= len(pos) else (0 if max_scans == 0 else len(self.base))

    def scores64(self, Q):
        if self.metric == orc.COSINE and self._xn is None:
            self._xn = _fp32_norms(self.base)
        return f64_scores(self.base, Q, self.metric, self._xn)

    def check(self, Q, k, max_scans=-1, ctx="", want=None, S=None):
        """Search both, run both checks; returns the GPU result.  want / S: the oracle's result and scores64(Q), when
        already at hand."""
        got = _s(self.ix, Q, k, max_scans=max_scans)
        if want is None:
            want = self.ref.search_batch(Q, k, max_scans=max_scans, nthreads=NT)
        assert_batch_equivalent(want, got, ctx=ctx)
        if self.ix.kind != self.pg.FLAT or _kernel(self.ix).startswith("flat_tc_kernel"):
            # tensor-core candidates are re-scored in the reference's arithmetic: bit for bit where the ids agree (the
            # CUDA-core scan sums in its own order and is held to the 1e-4 bar alone)
            same = want[0] == got[0]
            np.testing.assert_array_equal(want[1][same], got[1][same], err_msg=f"{ctx}: scores of agreeing ids differ")
        S = self.scores64(Q) if S is None else S
        f64_check(self.base, self.live, self.cutoff(max_scans), Q, self.metric, got, S=S, ctx=ctx)
        return got


def _kernel(ix):
    return ix.last_search_kernel()[0]


def assert_regime(ix, regime, ctx=""):
    """regime: '3x' | 'twopass' | 'fp16' | 'tf32' | 'cuda' (the CUDA-core scan, which names no kernel).
    The two 3xTF32 regimes differ by the pass-A, select and pass-B launches: a single pass takes at most 6 (query norms,
    query split, operand prepare, scan, re-score, merge), the two-pass path at least 7."""
    name, launches = _kernel(ix), ix.last_search_launches()
    if regime == "cuda":
        assert not name.startswith("flat_tc_kernel"), f"{ctx}: expected the CUDA-core scan, got {name!r}"
    elif regime == "3x":
        assert name == K3X and launches <= 6, f"{ctx}: expected one 3xTF32 pass, got {name!r} with {launches} launches"
    elif regime == "twopass":
        assert name == K3X and launches >= 7, f"{ctx}: expected the two-pass path, got {name!r} with {launches} launches"
    else:
        want = KF16 if regime == "fp16" else KTF32
        assert name == want, f"{ctx}: expected {want!r}, got {name!r}"


def expected_regime(dim, n_scan, k, metric, f16_table=True):
    """The dispatch table above, as the tests expect it."""
    kp = k + (16 if k < 64 else 32)
    if kp > 224 or n_scan < 8192:
        return "cuda"
    if dim > 256 and n_scan >= 65536:
        return "fp16" if (metric != orc.COSINE and dim % 8 == 0 and f16_table) else "tf32"
    if dim <= 256 and n_scan >= 16384 and kp >= 32:
        return "twopass"
    return "3x"


_CACHE = {}


@pytest.fixture(scope="module")
def pairs(gpu):
    """One index per (shape, metric), built on first use and kept for the module."""
    def get(n, d, metric, seed=1):
        key = (n, d, metric, seed)
        if key not in _CACHE:
            _CACHE[key] = Pair(gpu, metric, _data(n, d, seed))
        return _CACHE[key]
    yield get
    for p in _CACHE.values():
        p.ix.close()
    _CACHE.clear()


# ------------------------------------------------------------------------------------------------
# 1. the regime matrix
# ------------------------------------------------------------------------------------------------
MATRIX = [
    ("twopass", 20_000, 128, "L2"), ("twopass", 20_000, 128, "IP"), ("twopass", 20_000, 128, "COSINE"),
    ("fp16", 70_001, 320, "L2"), ("fp16", 70_001, 320, "IP"),                     # rows not a multiple of BN = 256
    ("tf32", 70_001, 260, "L2"), ("tf32", 70_001, 260, "IP"),                     # d % 8 != 0, K not a multiple of 32
    ("tf32", 70_001, 320, "COSINE"),
    ("3x", 60_000, 320, "L2"), ("3x", 60_000, 320, "IP"), ("3x", 60_000, 320, "COSINE"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("regime,n,d,metric", MATRIX, ids=[f"{r}-{n}x{d}-{m}" for r, n, d, m in MATRIX])
def test_regime_matrix(pairs, regime, n, d, metric):
    """nq 1 / 129 / 300: odd and even query-tile counts (a padded cluster partner) and many row splits."""
    p = pairs(n, d, METRICS[metric])
    Q = _queries(300, d, n + d)
    S = p.scores64(Q)
    for k in (1, 10, 100):
        want = p.ref.search_batch(Q, k, nthreads=NT)
        for nq in (1, 129, 300):
            ctx = f"{regime} {n}x{d} {metric} nq={nq} k={k}"
            p.check(Q[:nq], k, ctx=ctx, want=tuple(a[:nq] for a in want), S=S[:nq])
            exp = expected_regime(d, n, k, METRICS[metric])
            assert exp == regime or (regime == "twopass" and k < 16 and exp == "3x"), ctx
            assert_regime(p.ix, exp, ctx)


# ------------------------------------------------------------------------------------------------
# 2. k at the limits
# ------------------------------------------------------------------------------------------------
KLIM = [("twopass", 20_000, 128, "L2"), ("fp16", 70_001, 320, "IP"), ("tf32", 70_001, 320, "COSINE"),
        ("3x", 60_000, 320, "L2")]


@pytest.mark.gpu
@pytest.mark.parametrize("regime,n,d,metric", KLIM, ids=[f"{r}-{m}" for r, n, d, m in KLIM])
def test_k_limits(pairs, regime, n, d, metric):
    """k 15 / 16 (k' 31 / 32: the two-pass switch), 63 / 64 (margin 16 / 32), 192 (k' = 224, queue cap 512) with few
    queries, so many splits overfill the re-score window and it takes several rounds; 193 leaves the tensor cores."""
    p = pairs(n, d, METRICS[metric])
    Q = _queries(129, d, 7 * n + d)
    for k, nq in ((15, 129), (16, 129), (63, 129), (64, 129), (192, 4), (192, 1), (193, 4)):
        ctx = f"{regime} {metric} k={k} nq={nq}"
        p.check(Q[:nq], k, ctx=ctx)
        assert_regime(p.ix, expected_regime(d, n, k, METRICS[metric]), ctx)
    assert expected_regime(d, n, 193, METRICS[metric]) == "cuda"


# ------------------------------------------------------------------------------------------------
# 3. row-count and MaxScans switches, tombstones, upserts, appends
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,d,k,metric", [(8191, 128, 10, "L2"), (8192, 128, 10, "IP"),
                                          (16_383, 128, 100, "L2"), (16_384, 128, 100, "COSINE"),
                                          (65_535, 320, 10, "IP"), (65_536, 320, 10, "L2")])
def test_row_count_switches(gpu, n, d, k, metric):
    p = Pair(gpu, METRICS[metric], _data(n, d, 3))
    Q = _queries(130, d, n)
    p.check(Q, k, ctx=f"n={n} d={d} k={k} {metric}")
    assert_regime(p.ix, expected_regime(d, n, k, METRICS[metric]), f"n={n}")
    p.ix.close()


def _ms_for_cutoff(p, cut):
    """max_scans that puts the scan cut-off at exactly `cut` (row cut - 1 must be live)."""
    assert p.live[cut - 1]
    return int(p.live[:cut].sum())


@pytest.mark.gpu
@pytest.mark.parametrize("n,d,metric,k,switches", [
    (70_000, 320, "L2", 10, (65_536, 8192)),       # fp16 one-term / 3xTF32 / CUDA core
    (20_000, 128, "IP", 100, (16_384, 8192)),      # two-pass / 3xTF32 / CUDA core
])
def test_tombstones_maxscans_upserts_appends(gpu, n, d, metric, k, switches):
    rng = np.random.default_rng(n + 5)
    p = Pair(gpu, METRICS[metric], _data(n, d, 4))
    Q = _queries(64, d, n + 5)
    keep = set()
    for s in switches:
        keep |= {s - 2, s - 1, s}
    lo = switches[0]
    dels = [int(r) for r in rng.choice(lo, 3000, replace=False) if int(r) not in keep]
    for r in dels:
        p.delete(r)

    def sweep(tag):
        p.check(Q, k, ctx=f"{tag} full")
        assert_regime(p.ix, expected_regime(d, len(p.base), k, p.metric), f"{tag} full")
        for s in switches:
            for cut in (s - 1, s):
                ms = _ms_for_cutoff(p, cut)
                assert p.cutoff(ms) == cut
                ctx = f"{tag} max_scans={ms} (n_scan {cut})"
                p.check(Q, k, max_scans=ms, ctx=ctx)
                assert_regime(p.ix, expected_regime(d, cut, k, p.metric), ctx)

    sweep("tombstones")
    live = np.flatnonzero(p.live)
    for r in rng.choice(live[live < lo], 200, replace=False):          # in-place upserts below the switch
        p.update(int(r), (Q[int(r) % len(Q)] * np.float32(1.5)).astype(np.float32) if r % 4 == 0 else
                 rng.standard_normal(d, dtype=np.float32))
    p.append(rng.standard_normal((1000, d), dtype=np.float32))
    sweep("upserts + appends")
    p.ix.close()


@pytest.mark.gpu
def test_growth_across_the_fp16_switch(gpu):
    """3xTF32 at 60,000 rows; fp16 one-term after appending to 70,000; a row beyond fp16 (32,768.004) turns it to
    1xTF32; writing that component back to 1.0 reconverts from row 0 and returns to fp16; a row at exactly 32,768
    stays fp16."""
    d = 320
    full = _data(70_000, d, 6)
    p = Pair(gpu, orc.L2, full[:60_000])
    Q = _queries(129, d, 6)
    p.check(Q, 10, ctx="60,000 rows")
    assert_regime(p.ix, "3x", "60,000 rows")
    p.append(full[60_000:])
    p.check(Q, 10, ctx="70,000 rows")
    assert_regime(p.ix, "fp16", "70,000 rows")
    big = _data(1, d, 7)[0]
    big[5] = np.float32(32768.004)
    assert big[5] > 32768.0
    p.append(big)
    Q[3] = big                                                            # its own best match
    p.check(Q, 10, ctx="a row beyond fp16")
    assert_regime(p.ix, "tf32", "a row beyond fp16")
    assert p.ix.last_search_kernel()[0] == KTF32
    fixed = big.copy()
    fixed[5] = np.float32(1.0)
    p.update(70_000, fixed)
    p.check(Q, 10, ctx="written back to 1.0")
    assert_regime(p.ix, "fp16", "written back to 1.0")
    edge = _data(1, d, 8)[0]
    edge[9] = np.float32(32768.0)
    p.append(edge)
    Q[4] = edge
    p.check(Q, 10, ctx="a row at exactly 32,768")
    assert_regime(p.ix, "fp16", "a row at exactly 32,768")
    p.ix.close()


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["L2", "IP"])
def test_band_overflow_from_near_ties(gpu, metric):
    """1,000 exact duplicates of a row c whose values fp16 holds exactly, and a ladder of 600 rows c + t s (t in (0, 1])
    later in the scan that scores better than the duplicates, queries on top of them.  More than cap - 64 candidates sit
    inside the band, so the one-term queue overflows and keeps only k' of them, chosen by an fp16 proxy that cannot rank
    them: for IP (s = 2e-4) the ladder rounds to c's own fp16 copy, for L2 (s = 2e-2, queries at c + 3e-2, one rung
    2e-4 apart in score: within reach of the three-term pass, not of fp16's rounding).  Only the three-term pass behind,
    which redoes the batch, finds the true top k."""
    rng = np.random.default_rng(21)
    d = 320
    base = rng.random((70_001, d), dtype=np.float32)
    c = (np.float32(0.5) + np.float32(0.5) * rng.random(d, dtype=np.float32)).astype(np.float16).astype(np.float32)
    base[1000:2000] = c
    t = (np.arange(1, 601, dtype=np.float32) / np.float32(600))[:, None]
    Q = rng.random((40, d), dtype=np.float32)
    if metric == "IP":
        base[30_000:30_600] = c + t * np.float32(2e-4)
        assert (base[30_000:30_600].astype(np.float16).astype(np.float32) == c).all()
        Q[:8] = c + rng.random((8, d), dtype=np.float32) * np.float32(1e-4)
    else:
        base[30_000:30_600] = c + t * np.float32(2e-2)
        Q[:8] = c + np.float32(3e-2)
    Q[8] = c
    p = Pair(gpu, METRICS[metric], base)
    for k, nq in ((10, 40), (192, 4), (192, 40)):
        got = p.check(Q[:nq], k, ctx=f"near ties {metric} k={k} nq={nq}")
        assert_regime(p.ix, "fp16", f"near ties k={k}")
        assert (got[0][0, :k] >= 30_000 + 600 - k - 1).all()      # the ladder's best, above every duplicate
    p.ix.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scale,metric", [(3e-5, "IP"), (2e-7, "IP"), (2e-7, "L2")])
def test_fp16_subnormal_table(gpu, scale, metric):
    """Every value below fp16's smallest normal (6.1e-5), or around its smallest subnormal (6e-8), where the copies
    hold a few ulps or 0: the band must carry the absolute rounding error of the subnormals.  Scores of the 2e-7
    table are ~1e-12, far below the oracle comparison's absolute tolerance: the float64 check carries this case."""
    rng = np.random.default_rng(22)
    base = (rng.random((70_001, 320), dtype=np.float32) * np.float32(scale)).astype(np.float32)
    p = Pair(gpu, METRICS[metric], base)
    Q = (rng.random((300, 320), dtype=np.float32) * np.float32(scale)).astype(np.float32)
    for k in (10, 100):
        p.check(Q, k, ctx=f"subnormal {scale} {metric} k={k}")
        assert_regime(p.ix, "fp16", "subnormal")
    p.ix.close()


# ------------------------------------------------------------------------------------------------
# 4. cosine rows at the 1e-6 norm cut
# ------------------------------------------------------------------------------------------------
def _lane_strided_norm(x):
    """|x| summed the way a warp sums it: lane-strided fma, then an xor butterfly (float64 product, one rounding)."""
    acc = np.zeros(32, np.float32)
    for i, v in enumerate(np.asarray(x, np.float32)):
        acc[i % 32] = np.float32(np.float64(v) * np.float64(v) + np.float64(acc[i % 32]))
    for o in (16, 8, 4, 2, 1):
        acc = (acc + acc[np.arange(32) ^ o]).astype(np.float32)
    return np.float32(np.sqrt(acc[0]))


def _below_cut_row(u):
    """A row close to direction u whose reference norm is below 1e-6 but whose norm summed in another order is not."""
    rng = np.random.default_rng(0)
    cut = np.float32(1e-6)
    for _ in range(400):
        for j in range(0, -8, -1):
            x = (u * np.float32(1e-6 * (1 + j * 2.0 ** -23))).astype(np.float32)
            if np.float32(orc.norm(x)) < cut <= _lane_strided_norm(x):
                return x
        u = np.abs(u * (1 + np.float32(1e-3) * rng.standard_normal(len(u), dtype=np.float32))).astype(np.float32)
        u = (u / np.float32(np.linalg.norm(u))).astype(np.float32)
    return None


def _cosine_cut_table(n, d, seed):
    rng = np.random.default_rng(seed)
    base = rng.random((n, d), dtype=np.float32)
    q = rng.random(d, dtype=np.float32)
    u = (q / np.float32(np.linalg.norm(q))).astype(np.float32)
    ladder = np.array([(u * np.float32(1e-6 * (1 + j * 2.0 ** -23))).astype(np.float32) for j in range(-1000, 1001)])
    base[500:2501] = ladder
    base[3000] = 0.0
    base[3001] = rng.random(d, dtype=np.float32) * np.float32(1e4 / np.sqrt(d / 3.0))
    v = rng.random(d, dtype=np.float32) ** 4                         # a direction no random row is close to
    v = (v / np.float32(np.linalg.norm(v))).astype(np.float32)
    crowd = _below_cut_row(v)
    assert crowd is not None, "no row found on the edge of the cut"
    base[4000:4300] = crowd                                         # 300 rows that score 0, pointing at query 1
    Q = rng.random((8, d), dtype=np.float32)
    Q[0] = q
    Q[1] = v
    Q[2] = (u * np.float32(5e-7)).astype(np.float32)                 # query norm below 1e-6: every score is 0
    Q[3] = ladder[1000]
    return base, Q


COSCUT = [("3x", 60_000, 320), ("twopass", 20_000, 128), ("tf32", 70_001, 320)]


@pytest.mark.gpu
@pytest.mark.parametrize("regime,n,d", COSCUT, ids=[c[0] for c in COSCUT])
def test_cosine_rows_at_the_norm_cut(gpu, regime, n, d):
    """A ladder of 2,001 rows along a query's direction with norms 1e-6 (1 + j 2^-23), j in [-1000, 1000]; a zero row; a
    row of norm 1e4; 300 copies of a row just below the cut (score 0) pointing at another query; a query below the
    cut.  The zero-or-not decision must be the reference's, taken on the exact norm, in every pass."""
    base, Q = _cosine_cut_table(n, d, n)
    p = Pair(gpu, orc.COSINE, base)
    live = int(p.live.sum())
    for k in (10, 100, 192):
        got = p.check(Q, k, ctx=f"cosine cut {regime} k={k}")
        assert_regime(p.ix, expected_regime(d, n, k, orc.COSINE), f"cosine cut {regime} k={k}")
        assert int(got[2][2]) == min(k, live) and (got[1][2][:k] == 0).all()
        assert 3000 not in got[0][0] and not np.isin(got[0][1], np.arange(4000, 4300)).any()
    p.ix.close()


# ------------------------------------------------------------------------------------------------
# 5. IVF_FLAT write buffer: the same one-term regime in the IvfFlat evaluation order
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["COSINE", "IP"])
def test_ivf_flat_write_buffer_one_term(gpu, metric):
    base = _data(70_001, 320, 11)
    p = Pair(gpu, METRICS[metric], base, kind=gpu.IVF_FLAT)
    assert not p.ix.is_built()
    Q = _queries(129, 320, 11)
    for k in (10, 100):
        p.check(Q, k, ctx=f"IVF_FLAT buffer {metric} k={k}")
        # query norms (cosine), query split, band + scan, (fp16 query copy), scan + re-score, merge: a 3xTF32 pass
        # would take 4 (5 with cosine)
        assert p.ix.last_search_launches() >= 7
    p.ix.close()


# ------------------------------------------------------------------------------------------------
# 6. switches: per-search ones in-process, process-wide ones in a child process
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("var,case", [("PYROPE_TC_3X", ("fp16", 70_001, 320, "L2")),
                                      ("PYROPE_TC_3X", ("tf32", 70_001, 320, "COSINE")),
                                      ("PYROPE_TC_PASSA_3X", ("twopass", 20_000, 128, "IP")),
                                      ("PYROPE_TC_PASSB_3X", ("twopass", 20_000, 128, "L2"))])
def test_per_search_switches(pairs, monkeypatch, var, case):
    regime, n, d, metric = case
    p = pairs(n, d, METRICS[metric])
    Q = _queries(129, d, 99)
    a = p.check(Q, 100, ctx=f"{case} default")
    assert_regime(p.ix, regime, "default")
    monkeypatch.setenv(var, "1")
    b = p.check(Q, 100, ctx=f"{case} {var}")
    assert_regime(p.ix, "3x" if var == "PYROPE_TC_3X" else "twopass", var)
    monkeypatch.delenv(var)
    assert_batch_equivalent(a, b, ctx=f"{var} vs default")
    same = a[0] == b[0]
    np.testing.assert_array_equal(a[1][same], b[1][same])


def _fp16_case_data():
    return _data(70_001, 320, 1), _queries(640, 320, 70_001 + 320)


def child_flat_fp16(out, nqs=(129,), k=100):
    """Child-process side: build the fp16 one-term L2 case from its seed and save the searches."""
    import pyrope_b200 as pg
    pg._lib.check(pg.load().pyrope_gpu_init(0))
    base, Q = _fp16_case_data()
    ix = pg.GpuIndex(pg.FLAT, 320, pg.L2)
    ix.add(base)
    res = {}
    for nq in nqs:
        rows, sc, cnt = _s(ix, Q[:nq], k)
        res.update({f"rows{nq}": rows, f"scores{nq}": sc, f"counts{nq}": cnt,
                    f"kernel{nq}": np.array(_kernel(ix))})
    np.savez(out, **res)


@pytest.fixture()
def in_child(tmp_path):
    """run(env, "module:function", **kwargs): call the function in a fresh interpreter with `env` added to the
    environment, passing it an .npz path under tmp_path; returns the loaded arrays.  subprocess.run waits for the
    child; a non-zero exit fails the test with the child's stderr in the captured output."""
    count = [0]

    def run(env, target, **kwargs):
        mod, fn = target.split(":")
        count[0] += 1
        out = str(tmp_path / f"child{count[0]}.npz")
        code = (f"import sys; sys.path.insert(0, {ROOT!r}); import importlib; "
                f"importlib.import_module({mod!r}).{fn}({out!r}, **{kwargs!r})")
        full = dict(os.environ)
        full.update(env)
        args = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
        subprocess.run(args, env=full, cwd=ROOT, timeout=900, check=True)
        with np.load(out) as z:
            return {key: z[key] for key in z.files}

    return run


@pytest.mark.gpu
@pytest.mark.parametrize("env,nqs,kernel", [
    ({"PYROPE_FLAT_TF32": "1"}, (129,), KTF32),
    ({"PYROPE_FLAT_NOCLUSTER": "1"}, (129, 300), KF16),
    ({"PYROPE_FLAT_CLUSTER": "4"}, (100, 300, 600), KF16),        # 1, 3 and 5 query tiles: padded clusters of 4
], ids=["flat_tf32", "nocluster", "cluster4"])
def test_process_wide_switches(pairs, in_child, env, nqs, kernel):
    p = pairs(70_001, 320, orc.L2)
    base, Q = _fp16_case_data()
    np.testing.assert_array_equal(base, p.base)
    child = in_child(env, "tests.test_gpu_flat_tc_regimes:child_flat_fp16", nqs=nqs, k=100)
    for nq in nqs:
        ctx = f"{env} nq={nq}"
        assert str(child[f"kernel{nq}"]) == kernel, ctx
        got = (child[f"rows{nq}"], child[f"scores{nq}"], child[f"counts{nq}"])
        default = p.check(Q[:nq], 100, ctx=f"default nq={nq}")
        assert_regime(p.ix, "fp16", "default")
        assert_batch_equivalent(default, got, ctx=f"{ctx} vs default")
        same = default[0] == got[0]
        np.testing.assert_array_equal(default[1][same], got[1][same])
        want = p.ref.search_batch(Q[:nq], 100, nthreads=NT)
        assert_batch_equivalent(want, got, ctx=f"{ctx} vs oracle")
        f64_check(p.base, p.live, len(p.base), Q[:nq], orc.L2, got, S=p.scores64(Q[:nq]), ctx=ctx)
