"""The list-major IVF_FLAT scan (ivf_lm.cu) and the coarse re-rank (build.cu: coarse_rerank_kernel) where fp32 sums
cancel, checked twice:

- against the oracle, which adopts the GPU index's own centroids and lists (so a mismatch points at the search, not at
  training): counts equal; for the list-major scan also ids equal modulo ties and scores bit-identical where the ids
  agree, on every data regime (the query-major kernel, which ranks in its own fp32 order, where scores are not near 0);
- against a float64 reference of the lists each query probed (f64_check_probed): the count is min(k, live probed
  rows), every returned score is its row's float64 score and no probed live row left out scores above the k-th
  returned one.  Tolerance: 1e-4 |s| plus the fp32 summation bound 4 ulp x d x (|q| max|x| for IP, (|q| + max|x|)^2
  for L2, 1 for cosine).

Batches of >= 64 queries take the list-major kernels, 63 the query-major one (ivf.cu), on the same data.  The data
regimes put the k-th score where the seed's, the scan's and the reference's summation orders disagree by more than a
margin relative to the score: rows orthogonal to the queries' span (every score is rounding noise), zero-mean rows,
magnitudes 1e-3 .. 1e3 inside a row, exact duplicates spread over several lists."""
import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.parity import assert_batch_equivalent
from tests.test_gpu_flat_tc_regimes import f64_check, f64_scores

NT = orc.max_threads()
METRICS = {"L2": orc.L2, "IP": orc.IP, "COSINE": orc.COSINE}
LM = "ivf_lm_scan_kernel"


# ------------------------------------------------------------------------------------------------
# float64 reference over the probed lists
# ------------------------------------------------------------------------------------------------
def probe_lists(centroids, Q, metric, P):
    """[nq][P] lists each query probes, ranked by float64 scores (ties to the lower index).  The tables below keep the
    centroid scores far apart, so this is the reference's fp32 ranking too."""
    S = f64_scores(centroids, Q, metric)
    return np.argsort(-S, axis=1, kind="stable")[:, :P]


def probed_mask(probes, list_off, list_rows, n):
    """[nq][n] bool: the rows of the lists each query probed (-1 entries probe nothing)."""
    m = np.zeros((len(probes), n), bool)
    for q, ls in enumerate(probes):
        for l in ls:
            if l >= 0:
                m[q, list_rows[list_off[l]:list_off[l + 1]]] = True
    return m


def f64_check_probed(base, live, probes, list_off, list_rows, Q, metric, got, S=None, ctx=""):
    """f64_check per query, its live mask the live rows of the lists that query probed."""
    base = np.asarray(base, np.float32)
    S = f64_scores(base, Q, metric) if S is None else S
    mask = probed_mask(probes, list_off, list_rows, len(base)) & np.asarray(live, bool)[None, :]
    rows, sc, cnt = got
    for q in range(len(Q)):
        f64_check(base, mask[q], len(base), Q[q:q + 1], metric, (rows[q:q + 1], sc[q:q + 1], cnt[q:q + 1]),
                  S=S[q:q + 1], ctx=f"{ctx} (query {q})")


def test_f64_check_probed_accepts_oracle_and_rejects_a_dropped_row():
    """CPU: the per-query check agrees with the oracle's IVF_FLAT search on all three metrics (lists adopted, deletes
    included), and flags a result whose best row was removed."""
    rng = np.random.default_rng(4)
    n, d, nlist, P = 600, 20, 12, 6
    base = (rng.standard_normal((n, d)) * 2).astype(np.float32)
    Q = rng.standard_normal((10, d)).astype(np.float32)
    cent = (rng.standard_normal((nlist, d)) * 3).astype(np.float32)
    assign = np.argmax(f64_scores(base, cent, orc.L2), axis=0)   # nearest centroid (lists only need to be a partition)
    list_rows = np.argsort(assign, kind="stable")
    off = np.searchsorted(assign[list_rows], np.arange(nlist + 1))
    live = np.ones(n, bool)
    live[rng.choice(n, 50, replace=False)] = False
    for name, metric in METRICS.items():
        ref = orc.IvfFlatIndex(d, metric, nlist=nlist)
        ref.adopt(cent, off, list_rows, base[list_rows])
        for r in np.flatnonzero(~live):
            assert ref.delete(int(r))
        probes = probe_lists(cent, Q, metric, P)
        got = ref.search_batch(Q, 10, nprobe=P, nthreads=NT)
        f64_check_probed(base, live, probes, off, list_rows, Q, metric, got, ctx=f"oracle {name}")
        rid, rsc, rcn = ref.search_batch(Q, 11, nprobe=P, nthreads=NT)
        assert (rcn == 11).all()
        bad = (rid[:, 1:].copy(), rsc[:, 1:].copy(), np.minimum(rcn, 10))
        with pytest.raises(AssertionError, match="missing row"):
            f64_check_probed(base, live, probes, off, list_rows, Q, metric, bad, ctx=f"dropped {name}")
        short = (rid[:, :10].copy(), rsc[:, :10].copy(), np.minimum(rcn, 9))
        with pytest.raises(AssertionError, match="count"):
            f64_check_probed(base, live, probes, off, list_rows, Q, metric, short, ctx=f"short {name}")


# ------------------------------------------------------------------------------------------------
# data regimes
# ------------------------------------------------------------------------------------------------
def _span_basis(d, r, rng):
    """An orthonormal basis (float64, [d][r]) of an r-dimensional subspace and one of its complement ([d][d - r])."""
    B, _ = np.linalg.qr(rng.standard_normal((d, d)))
    return B[:, :r], B[:, r:]


def make_data(kind, n, d, nq, seed):
    """(rows [n][d], queries [nq][d]) of one regime."""
    rng = np.random.default_rng(seed)
    if kind == "uniform":                                     # every product positive: nothing cancels
        return rng.random((n, d), dtype=np.float32), rng.random((nq, d), dtype=np.float32)
    if kind == "zero_mean":
        return rng.standard_normal((n, d), dtype=np.float32), rng.standard_normal((nq, d), dtype=np.float32)
    if kind == "orthogonal":                                  # queries in an r-dim subspace, rows in its complement x 100
        r = max(1, min(8, d // 2))
        span, comp = _span_basis(d, r, rng)
        Q = (rng.standard_normal((nq, r)) @ span.T).astype(np.float32)
        X = (100.0 * rng.standard_normal((n, d - r)) @ comp.T).astype(np.float32)
        return X, Q
    if kind == "mixed":                                       # magnitudes 1e-3 .. 1e3 inside one row
        mag = (10.0 ** rng.uniform(-3, 3, d)).astype(np.float32)
        X = (rng.standard_normal((n, d), dtype=np.float32) * mag).astype(np.float32)
        Q = (rng.standard_normal((nq, d), dtype=np.float32) * mag[::-1]).astype(np.float32)
        return X, Q
    if kind == "duplicates":
        # 24 distinct rows, each repeated, queries near some.  The queries are 0 in the last dimension and the copies hold
        # +-c there: +c and -c copies tie exactly on every metric (same products, same norm) and the large last
        # component sends them to different lists (test_regimes checks that the ties are spread)
        U = rng.standard_normal((24, d), dtype=np.float32)
        X = U[rng.integers(0, 24, n)]
        Q = (U[rng.integers(0, 24, nq)] + np.float32(0.05) * rng.standard_normal((nq, d), dtype=np.float32))
        X[:, -1] = np.float32(3 * np.sqrt(d)) * rng.choice(np.array([-1, 1], np.float32), n)
        Q[:, -1] = 0.0
        return X.astype(np.float32), Q.astype(np.float32)
    raise ValueError(kind)


def make_centroids(X, Q, nlist, seed):
    """Frozen centroids whose scores against every query are far apart (the coarse stage is not under test here): a
    random direction per list plus a component along the mean query, scaled to the rows."""
    rng = np.random.default_rng(seed + 17)
    d = X.shape[1]
    scale = float(np.sqrt((X.astype(np.float64) ** 2).sum(1).mean() / d)) or 1.0
    C = rng.standard_normal((nlist, d)) * scale
    qm = Q.astype(np.float64).mean(0)
    qm /= np.linalg.norm(qm) or 1.0
    C += np.linspace(-3, 3, nlist)[:, None] * scale * np.sqrt(d) * qm[None, :]
    return C.astype(np.float32)


# ------------------------------------------------------------------------------------------------
# GPU pair
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


def lm_expected(nq, d, P, k):
    """The dispatch of the list-major scan: >= 64 queries, d % 4 == 0, d <= 1,024, P k <= 16,384, no budget."""
    return nq >= 64 and d % 4 == 0 and 4 <= d <= 1024 and 1 <= k <= 1024 and P * k <= 16384


class IvfPair:
    """A GPU IVF_FLAT index over frozen centroids next to the oracle's, which adopts the GPU's lists."""

    def __init__(self, pg, metric, base, centroids, query_major_strict=False):
        self.pg, self.metric, self.qm_strict = pg, metric, query_major_strict
        self.base = np.array(base, np.float32)
        self.cent = np.array(centroids, np.float32)
        n, d = self.base.shape
        self.live = np.ones(n, bool)
        self.ix = pg.GpuIndex(pg.IVF_FLAT, d, _gm(pg, metric), nlist=len(self.cent))
        self.ix.set_codebooks(self.cent)
        self.ix.add(self.base)
        self.ix.build()
        self.off, self.rows, _ = self.ix.lists()
        assert self.off[-1] == n
        self.ref = orc.IvfFlatIndex(d, metric, nlist=len(self.cent))
        self.ref.adopt(self.cent, self.off, self.rows, self.base[self.rows])

    def delete(self, row):
        assert self.ref.delete(int(row)) and self.ix.delete_row(int(row))
        self.live[row] = False

    def list_len(self):
        return np.diff(self.off)

    def check(self, Q, k, P, ctx="", S=None):
        got = _s(self.ix, Q, k, nprobe=P)
        name = self.ix.last_search_kernel()[0]
        want_lm = lm_expected(len(Q), Q.shape[1], P, k)
        assert (name == LM) == want_lm, f"{ctx}: kernel {name!r}, list-major expected: {want_lm}"
        want = self.ref.search_batch(Q, k, nprobe=P, nthreads=NT)
        if want_lm:
            # ranked and re-scored in the reference's order: its rows (modulo ties) and its scores, bit for bit
            assert_batch_equivalent(want, got, ctx=ctx)
            same = want[0] == got[0]
            np.testing.assert_array_equal(want[1][same], got[1][same], err_msg=f"{ctx}: scores of agreeing ids differ")
        elif self.qm_strict:
            # the query-major kernel ranks and scores in its own fp32 order: held to the oracle's 1e-4 bar where scores are
            # not near 0 (elsewhere its 1e-6 absolute part is below the rounding of the sums), always to the counts and
            # the float64 check below
            assert_batch_equivalent(want, got, ctx=ctx)
        np.testing.assert_array_equal(want[2], got[2], err_msg=f"{ctx}: counts differ")
        probes = probe_lists(self.cent, Q, self.metric, P)
        f64_check_probed(self.base, self.live, probes, self.off, self.rows, Q, self.metric, got, S=S, ctx=ctx)
        return got


def _pair(gpu, kind, metric, n, d, nlist, seed, nq=64):
    X, Q = make_data(kind, n, d, nq, seed)
    strict = kind == "uniform" or (metric == orc.L2 and kind != "orthogonal")
    return IvfPair(gpu, metric, X, make_centroids(X, Q, nlist, seed), query_major_strict=strict), Q


DIMS = [4, 64, 124, 128, 132, 768, 1020, 1024]
CASES = ([(d, m, "zero_mean") for d in DIMS for m in METRICS] + [(d, m, "orthogonal") for d in DIMS for m in METRICS] +
         [(d, m, kind) for d in (64, 132, 1020) for m in METRICS for kind in ("uniform", "mixed", "duplicates")])


@pytest.mark.gpu
@pytest.mark.parametrize("d,metric,kind", CASES, ids=[f"{k}-d{d}-{m}" for d, m, k in CASES])
def test_regimes(gpu, d, metric, kind):
    """3,000 rows over 32 lists.  nq 63 (query-major) and 64 (list-major) on the same queries; k = 1, 10, 100 with 4
    probes, 512 with 32 (every list: the seed samples 512 rows, P k = 16,384), 513 (no seed threshold)."""
    p, Q = _pair(gpu, kind, METRICS[metric], 3000, d, 32, seed=d * 7 + len(kind))
    if kind == "duplicates":                                     # exact ties in more than one list
        lists = np.repeat(np.arange(32), p.list_len())[np.argsort(p.rows)]
        key = [p.base[r, :-1].tobytes() for r in range(len(p.base))]
        spread = {}
        for r, kk in enumerate(key):
            spread.setdefault(kk, set()).add(int(lists[r]))
        assert max(len(v) for v in spread.values()) >= 2
    S = f64_scores(p.base, Q, p.metric)
    for k, P in ((1, 4), (10, 4), (100, 4), (512, 32), (513, 4)):
        for nq in (63, 64):
            p.check(Q[:nq], k, P, ctx=f"{kind} d={d} {metric} k={k} P={P} nq={nq}", S=S[:nq])
    p.ix.close()


@pytest.mark.gpu
@pytest.mark.parametrize("metric", list(METRICS))
@pytest.mark.parametrize("d", [64, 128, 132, 1024])
def test_k_covers_every_probed_row(gpu, d, metric):
    """300 rows orthogonal to the queries in 8 lists, all probed: k = 300 returns every row (the seed's sample covers
    them all, so its threshold must keep every one however the scan rounds), k = 299 all but the worst, and k =
    the longest list (no list is ever cut)."""
    p, Q = _pair(gpu, "orthogonal", METRICS[metric], 300, d, 8, seed=d + 1)
    S = f64_scores(p.base, Q, p.metric)
    for k in (300, 299, int(p.list_len().max()), 512):
        for nq in (63, 64):
            got = p.check(Q[:nq], k, 8, ctx=f"all rows d={d} {metric} k={k} nq={nq}", S=S[:nq])
            assert (got[2] == min(k, 300)).all()
    p.ix.close()


@pytest.mark.gpu
def test_dispatch_limit(gpu):
    """P k = 16,384 takes the list-major scan, 16,385 falls back to the query-major one: same answers."""
    p, Q = _pair(gpu, "zero_mean", orc.IP, 4000, 64, 40, seed=3)
    S = f64_scores(p.base, Q, p.metric)
    for k, P in ((512, 32), (565, 29), (1024, 16), (1, 40)):
        p.check(Q, k, P, ctx=f"limit k={k} P={P}", S=S)
    p.ix.close()


@pytest.mark.gpu
@pytest.mark.parametrize("nq", [15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129])
def test_query_groups_on_one_list(gpu, nq):
    """Every query probes the same list: 16 j and 16 j +- 1 queries make full and ragged 16-query work items."""
    X, Q = make_data("zero_mean", 2000, 132, 129, 8)
    p = IvfPair(gpu, orc.IP, X, X.mean(0, keepdims=True))   # one list holding every row
    for k in (1, 10, 300):
        p.check(Q[:nq], k, 1, ctx=f"one list nq={nq} k={k}")
    p.ix.close()


@pytest.mark.gpu
@pytest.mark.parametrize("metric", list(METRICS))
@pytest.mark.parametrize("d,ties", [(64, 300), (132, 300), (64, 2100), (768, 2100)])
def test_queue_overflow_and_ties(gpu, d, metric, ties):
    """`ties` exact copies of one row in one list, the queries on top of it: more than 256 candidates of one (query,
    list) overflow the scan's queue (the redo path); more than 2,048 fill the redo queue between prunes.  Ties keep
    the lower row, as the reference does."""
    rng = np.random.default_rng(d + ties)
    X = rng.standard_normal((ties + 1500, d), dtype=np.float32)
    X[:ties] = X[0]
    Q = (X[0] + np.float32(1e-3) * rng.standard_normal((64, d), dtype=np.float32)).astype(np.float32)
    C = rng.standard_normal((6, d), dtype=np.float32)
    C[0] = X[0]                                              # the copies' own list: every query probes it first
    p = IvfPair(gpu, METRICS[metric], X, C)
    assert p.list_len()[0] >= ties
    for k in (1, 10, 257, 1024):
        for nq in (63, 64):
            p.check(Q[:nq], k, 2, ctx=f"ties={ties} d={d} {metric} k={k} nq={nq}")
    p.ix.close()


@pytest.mark.gpu
@pytest.mark.parametrize("metric", list(METRICS))
@pytest.mark.parametrize("d", [64, 132])
def test_deletes_norm_cut_and_zero_query(gpu, d, metric):
    """Deleted rows (skipped by seed, scan and redo), cosine rows with norms just below and above 1e-6, a zero query."""
    rng = np.random.default_rng(d)
    X, Q = make_data("zero_mean", 3000, d, 64, d + 2)
    u = Q[1] / np.float32(np.linalg.norm(Q[1]))
    for j, f in enumerate((0.5, 0.999, 1.0, 1.001, 2.0)):
        X[10 + j] = (u * np.float32(1e-6 * f)).astype(np.float32)      # along query 1: norms around the cosine cut
    X[20] = 0.0
    Q[0] = 0.0
    p = IvfPair(gpu, METRICS[metric], X, make_centroids(X, Q, 16, d))
    for r in rng.choice(np.arange(30, 3000), 400, replace=False):
        p.delete(int(r))
    S = f64_scores(p.base, Q, p.metric)
    for k, P in ((10, 4), (300, 16), (600, 3)):
        for nq in (63, 64):
            got = p.check(Q[:nq], k, P, ctx=f"deletes d={d} {metric} k={k} P={P} nq={nq}", S=S[:nq])
            assert not np.isin(got[0], np.flatnonzero(~p.live)).any()
    p.ix.close()


@pytest.mark.gpu
@pytest.mark.parametrize("metric", list(METRICS))
@pytest.mark.parametrize("d", [64, 768])
def test_probes_supplied(gpu, d, metric):
    """Probes handed in through search_probed_device, with -1 entries and empty lists: the list scan apart from the
    coarse stage.  Reported scores are the reference's fp32 score of each row."""
    torch = pytest.importorskip("torch")
    X, Q = make_data("orthogonal", 2000, d, 96, d + 5)
    C = make_centroids(X, Q, 24, d)
    C[20:] = C[0]                                              # copies of list 0's centroid: ties go to list 0, empty lists
    p = IvfPair(gpu, METRICS[metric], X, C)
    assert (p.list_len()[20:] == 0).all()
    rng = np.random.default_rng(d)
    P = 6
    probes = np.stack([rng.permutation(24)[:P] for _ in range(len(Q))]).astype(np.int64)
    probes[::3, 2] = -1
    probes[::5, 0] = -1
    probes[7] = -1
    S = f64_scores(p.base, Q, p.metric)
    fn = {orc.L2: lambda a, b: -orc.l2sq(a, b), orc.IP: orc.dot, orc.COSINE: orc.cosine}[p.metric]
    ranked = []                                                 # per query: (score, list position, row) best first
    for q in range(len(Q)):
        c = [(np.float32(fn(Q[q], p.base[r])), pos, int(r)) for l in probes[q] if l >= 0
             for pos, r in enumerate(p.rows[p.off[l]:p.off[l + 1]], start=int(p.off[l]))]
        ranked.append(sorted(c, key=lambda t: (-float(t[0]), t[1])))

    def ref_topk(k):
        ids = np.full((len(Q), k), -1, np.int64)
        sc = np.zeros((len(Q), k), np.float32)
        cnt = np.zeros(len(Q), np.int32)
        for q, c in enumerate(ranked):
            cnt[q] = min(k, len(c))
            ids[q, :cnt[q]] = [t[2] for t in c[:k]]
            sc[q, :cnt[q]] = [t[0] for t in c[:k]]
        return ids, sc, cnt

    for k in (1, 50, 200):
        for nq in (63, 96):
            qd = torch.from_numpy(Q[:nq]).cuda()
            pd = torch.from_numpy(probes[:nq]).cuda()
            sc = torch.empty((nq, k), dtype=torch.float32, device="cuda")
            rw = torch.empty((nq, k), dtype=torch.int64, device="cuda")
            cn = torch.empty((nq,), dtype=torch.int32, device="cuda")
            st = torch.cuda.current_stream().cuda_stream
            p.ix.search_probed_device(qd.data_ptr(), nq, k, P, pd.data_ptr(), sc.data_ptr(), rw.data_ptr(),
                                      cn.data_ptr(), stream=st)
            torch.cuda.synchronize()
            got = (rw.cpu().numpy(), sc.cpu().numpy(), cn.cpu().numpy())
            ctx = f"probed d={d} {metric} k={k} nq={nq}"
            assert (p.ix.last_search_kernel()[0] == LM) == (nq >= 64), ctx
            f64_check_probed(p.base, p.live, probes[:nq], p.off, p.rows, Q[:nq], p.metric, got, S=S[:nq], ctx=ctx)
            if nq < 64:
                continue
            # the reference's ranking of the probed rows (VectorMath scores, ties to the earlier list position): on this
            # noise data the float64 check accepts almost any row, this pins membership
            assert_batch_equivalent(tuple(a[:nq] for a in ref_topk(k)), got, ctx=ctx)
            same = ref_topk(k)[0][:nq] == got[0]
            np.testing.assert_array_equal(ref_topk(k)[1][:nq][same], got[1][same], err_msg=f"{ctx}: scores differ")
    p.ix.close()


# ------------------------------------------------------------------------------------------------
# the coarse stage on small centroid tables: stage-one FLAT scan + coarse_rerank_kernel
# ------------------------------------------------------------------------------------------------
def oracle_probes(centroids, Q, metric, P):
    """The reference's ranking (IvfFlatVectorIndex.cs:186-198): VectorMath scores, descending, ties to the lower index."""
    fn = {orc.IP: orc.dot, orc.COSINE: orc.cosine, orc.L2: lambda a, b: -orc.l2sq(a, b)}[metric]
    out = np.zeros((len(Q), P), np.int64)
    for q in range(len(Q)):
        s = np.array([fn(Q[q], c) for c in centroids], np.float32)
        out[q] = np.lexsort((np.arange(len(s)), -s.astype(np.float64)))[:P]
    return out


def _coarse_table(nc, d, nq, seed):
    """nc centroids orthogonal to the queries' span (x 100: their scores are rounding noise around 0), 16 of them with a
    component along the queries; with P > 16 the P-th and (P+1)-th scores sit near 0, one query is 0."""
    rng = np.random.default_rng(seed)
    span, comp = _span_basis(d, 4, rng)
    Q = (rng.standard_normal((nq, 4)) @ span.T).astype(np.float32)
    Q[5] = 0.0
    C = 100.0 * rng.standard_normal((nc, d - 4)) @ comp.T
    C[:16] += rng.standard_normal((16, 4)) @ span.T
    return C.astype(np.float32), Q


def _coarse_index(gpu, kind, metric, C, X):
    d = C.shape[1]
    if kind == "IVF_FLAT":
        ix = gpu.GpuIndex(gpu.IVF_FLAT, d, _gm(gpu, metric), nlist=len(C))
        ix.set_codebooks(C)
    else:
        cb = np.random.default_rng(1).standard_normal((16, 256, d // 16), dtype=np.float32)
        ix = gpu.GpuIndex(gpu.IVF_PQ, d, _gm(gpu, metric), nlist=len(C), m=16, k=256)
        ix.set_codebooks(C, cb)
    ix.add(X)
    ix.build()
    return ix


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["IVF_FLAT", "IVF_PQ"])
@pytest.mark.parametrize("metric", ["IP", "COSINE"])
@pytest.mark.parametrize("nc,d", [(300, 64), (1500, 128), (1000, 768), (4096, 64)])
def test_coarse_probe_matches_reference_ranking(gpu, kind, metric, nc, d):
    """coarse_probe_device returns exactly the reference's probe sets; nc = 4,096 takes coarse_tc (the control), the
    smaller tables the stage-one FLAT scan and the re-rank gate.  IVF_FLAT, Cosine, small tables: a MaxScans budget walks
    the probed lists in the exact rank order (the budget forces the exact re-rank), checked through search against the
    oracle (IP: test_search_over_noise_centroids)."""
    torch = pytest.importorskip("torch")
    C, Q = _coarse_table(nc, d, 64, nc + d)
    X = np.random.default_rng(nc).standard_normal((4000, d), dtype=np.float32)
    om = METRICS[metric]
    ix = _coarse_index(gpu, kind, om, C, X)
    st = torch.cuda.current_stream().cuda_stream
    qd = torch.from_numpy(Q).cuda()
    for P in (1, 8, 20, 40):
        pd = torch.full((len(Q), P), -2, dtype=torch.int64, device="cuda")
        ix.coarse_probe_device(qd.data_ptr(), len(Q), P, pd.data_ptr(), stream=st)
        torch.cuda.synchronize()
        got = pd.cpu().numpy()
        want = oracle_probes(C, Q, om, P)
        bad = [q for q in range(len(Q)) if set(got[q]) != set(want[q])]
        assert not bad, f"{kind} {metric} nc={nc} P={P}: probe sets differ for queries {bad[:8]} ({len(bad)} of {len(Q)})"
    if kind == "IVF_FLAT" and metric == "COSINE" and nc < 2048:
        off, rows, _ = ix.lists()
        ref = orc.IvfFlatIndex(d, om, nlist=nc)
        ref.adopt(C, off, rows, X[rows])
        for P, ms in ((8, 40), (20, 200)):
            assert_batch_equivalent(ref.search_batch(Q, 10, nprobe=P, max_scans=ms, nthreads=NT),
                                    _s(ix, Q, 10, nprobe=P, max_scans=ms), ctx=f"budget {metric} nc={nc} P={P}")
    ix.close()


@pytest.mark.gpu
@pytest.mark.xfail(strict=True, reason="searches over these tables return other rows than the reference although "
                                       "coarse_probe_device returns the reference's probe sets; cause not yet found")
@pytest.mark.parametrize("metric,nc,d,budget", [("IP", 300, 64, True), ("IP", 4096, 64, False),
                                                ("COSINE", 4096, 64, False)])
def test_search_over_noise_centroids(gpu, metric, nc, d, budget):
    """IP with a MaxScans budget on a small table; IP and Cosine without one on a coarse_tc table."""
    C, Q = _coarse_table(nc, d, 64, nc + d)
    X = np.random.default_rng(nc).standard_normal((4000, d), dtype=np.float32)
    om = METRICS[metric]
    ix = _coarse_index(gpu, "IVF_FLAT", om, C, X)
    off, rows, _ = ix.lists()
    ref = orc.IvfFlatIndex(d, om, nlist=nc)
    ref.adopt(C, off, rows, X[rows])
    try:
        for P, ms in ((8, 40), (20, 200)):
            ms = ms if budget else -1
            assert_batch_equivalent(ref.search_batch(Q, 10, nprobe=P, max_scans=ms, nthreads=NT),
                                    _s(ix, Q, 10, nprobe=P, max_scans=ms), ctx=f"{metric} nc={nc} P={P} ms={ms}")
    finally:
        ix.close()


@pytest.mark.gpu
@pytest.mark.xfail(strict=True, reason="with coarse_tc (tables of >= 2,048 centroids) a MaxScans budget over IP centroid "
                                       "scores that are rounding noise walks other lists than the reference")
def test_coarse_tc_budget_order_on_noise_scores(gpu):
    C, Q = _coarse_table(4096, 64, 64, 4096 + 64)
    X = np.random.default_rng(4096).standard_normal((4000, 64), dtype=np.float32)
    ix = _coarse_index(gpu, "IVF_FLAT", orc.IP, C, X)
    off, rows, _ = ix.lists()
    ref = orc.IvfFlatIndex(64, orc.IP, nlist=4096)
    ref.adopt(C, off, rows, X[rows])
    assert_batch_equivalent(ref.search_batch(Q, 10, nprobe=8, max_scans=40, nthreads=NT),
                            _s(ix, Q, 10, nprobe=8, max_scans=40), ctx="coarse_tc budget")
    ix.close()
