"""The build path (build.cu: nearest_exact_kernel, assign_shortlist_kernel, kmeans_update_kernel; api.cu: assign_rows,
kmeans_train_device) bit for bit against the oracle where fp32 sums cancel.

"Centroid assignment and PQ code IDs must be bit-exact given the same trained codebooks": one row assigned to another
list changes the lists, every k-means iteration after it and every search result, and no search-side test can see it
(those make the oracle adopt the GPU's lists).  So coarse assignment, k-means, Build, Extend and PQ encoding are compared
with orc.find_nearest_centroid / orc.kmeans_train / IvfFlatIndex / IvfPqIndex / ProductQuantizer.encode, ties to the
lowest index, on data where the scores of many centroids are rounding noise: rows orthogonal to every centroid (IP scores
near 0 against |x||c| >= 1e4), rows 1e4 times longer than unit centroids they are orthogonal to (L2), zero-mean and
mixed-magnitude data, tiny values, crowds of exact copies of the winning centroid, zero rows and zero centroids.

At nlist >= 2,048 (d % 4 == 0) assignment shortlists k' = 17 centroids per row by 3xTF32 proxy scores and re-evaluates
them in the reference's order; a row whose shortlist cannot be proven complete is redone exhaustively.  The CPU tests
emulate that gate (emulate_shortlist) and check that the rounding-bound gate never accepts a shortlist missing the
oracle's winner while keeping almost every row of ordinary data, and that the margin it replaced (relative to the best
proxy plus 1e-4) accepts wrong shortlists in the orthogonal regimes, so the GPU cases there have teeth."""
import ctypes as C
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import pyoracle as orc
from tests.test_gpu_ivf_lm_regimes import _span_basis, make_data

NT = orc.max_threads()
KPRIME = 17                      # 1 + flat_tc_margin(1): the shortlist of assign_rows
METRICS = {"L2": orc.L2, "IP": orc.IP, "COSINE": orc.COSINE}
REGIMES = ["uniform", "zero_mean", "orthogonal", "mixed", "duplicates",
           "orth_ip_big", "sphere_l2", "tiny", "ties", "zeros"]


# ------------------------------------------------------------------------------------------------
# oracle, batched
# ------------------------------------------------------------------------------------------------
def oracle_assign(X, cent, metric):
    """orc.find_nearest_centroid for every row (the centroid norms computed once, rows on all cores)."""
    X = np.ascontiguousarray(X, np.float32)
    cent = np.ascontiguousarray(cent, np.float32)
    k, d = cent.shape
    cn = np.array([orc.norm(c) for c in cent], np.float32) if metric == orc.COSINE else np.zeros(k, np.float32)
    L, f32p = orc.lib(), C.POINTER(C.c_float)
    pc, pcn = cent.ctypes.data_as(f32p), cn.ctypes.data_as(f32p)
    rows = [X[i] for i in range(len(X))]
    with ThreadPoolExecutor(NT) as ex:
        out = ex.map(lambda r: L.orc_find_nearest_centroid(r.ctypes.data_as(f32p), pc, pcn, k, d, metric), rows)
        return np.fromiter(out, np.int32, len(X))


# ------------------------------------------------------------------------------------------------
# data regimes: (rows [n][d], centroids [nc][d])
# ------------------------------------------------------------------------------------------------
def _orth(n, nc, d, row_scale, rng, unit_centroids=False, cent_scale=1.0):
    """rows in an r-dim subspace, centroids in its complement: every exact score is ~0 (IP) or |x|^2 + |c|^2 (L2)."""
    r = max(1, min(8, d // 2))
    span, comp = _span_basis(d, r, rng)
    X = row_scale * rng.standard_normal((n, r)) @ span.T
    if comp.shape[1] == 0:                                   # d = 1: no complement, centroids along the row
        comp = span
    Cc = rng.standard_normal((nc, comp.shape[1])) @ comp.T
    if unit_centroids:
        Cc /= np.maximum(np.linalg.norm(Cc, axis=1, keepdims=True), 1e-30)
    return X.astype(np.float32), (cent_scale * Cc).astype(np.float32)


def assign_data(kind, n, nc, d, seed):
    rng = np.random.default_rng(seed)
    if kind in ("uniform", "zero_mean", "orthogonal", "mixed", "duplicates"):
        cent, X = make_data(kind, nc, d, n, seed)            # make_data's rows serve as centroids, its queries as rows
        return np.ascontiguousarray(X), np.ascontiguousarray(cent)
    if kind == "orth_ip_big":                                # |x| |c| ~ 1e4 .. 1e5, every IP score rounding noise
        return _orth(n, nc, d, 10.0, rng, cent_scale=1e3)
    if kind == "sphere_l2":                                  # |x| ~ 1e4 orthogonal to unit centroids: L2 ties to ~ulp(|x|^2)
        return _orth(n, nc, d, 1e4, rng, unit_centroids=True)
    if kind == "tiny":                                       # every score far below 1e-4
        return ((1e-3 * rng.standard_normal((n, d))).astype(np.float32),
                (1e-3 * rng.standard_normal((nc, d))).astype(np.float32))
    if kind == "ties":                                       # 40 > k' exact copies of the winner, the first one late
        cent = rng.standard_normal((nc, d)).astype(np.float32)
        copies = np.sort(rng.choice(np.arange(nc // 3, nc), 40, replace=False))
        cent[copies] = cent[copies[0]]
        X = (cent[copies[0]] + 0.01 * rng.standard_normal((n, d))).astype(np.float32)
        X[: n // 4] = cent[copies[0]]
        X[n // 2:] = rng.standard_normal((n - n // 2, d))
        return X, cent
    if kind == "zeros":                                      # zero rows and zero centroids (Cosine's 1e-6 norm cut)
        X = rng.standard_normal((n, d)).astype(np.float32)
        cent = rng.standard_normal((nc, d)).astype(np.float32)
        X[::7] = 0.0
        X[1::11] *= np.float32(1e-7)                          # |x| below the cut, not 0
        cent[3::5] = 0.0
        cent[4::9] *= np.float32(1e-7)
        return X, cent
    raise ValueError(kind)


# ------------------------------------------------------------------------------------------------
# CPU emulation of the shortlist and its gate
# ------------------------------------------------------------------------------------------------
def tf32_rn(x):
    """cvt.rna.tf32.f32: nearest, ties away from zero, 10 explicit mantissa bits."""
    b = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((b + 0x1000) & 0xFFFFE000).astype(np.uint32).view(np.float32)


def tf32_tr(x):
    """What kind::tf32 reads of an fp32 operand: the low 13 mantissa bits dropped."""
    return (np.asarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def proxy_terms(cent, metric):
    """(scale, bias) of tc_rowterms_kernel and A = max |scale_c| |c| of tc_amax_kernel (fp32)."""
    cent = np.asarray(cent, np.float32)
    sq = (cent.astype(np.float64) ** 2).sum(1).astype(np.float32)
    nrm = np.sqrt(sq)
    if metric == orc.L2:
        scale, bias = np.full(len(cent), 2, np.float32), -sq
    elif metric == orc.IP:
        scale, bias = np.ones(len(cent), np.float32), np.zeros(len(cent), np.float32)
    else:
        exact = np.array([orc.norm(c) for c in cent], np.float32)
        with np.errstate(divide="ignore"):
            scale = np.where((exact < 1e-6) | (nrm == 0), np.float32(0), np.float32(1) / nrm).astype(np.float32)
        bias = np.zeros(len(cent), np.float32)
    A = np.float32((np.abs(scale) * nrm).max())
    return scale, bias, A


def proxy_scores(X, cent, metric):
    """scale * (Xhi.Chi + Xhi.Clo + Xlo.Chi) + bias, the products summed in float64 (more accurate than the tensor
    pipe, so the emulation understates the proxy's error)."""
    X, cent = np.asarray(X, np.float32), np.asarray(cent, np.float32)
    xh, ch = tf32_rn(X), tf32_rn(cent)
    xl, cl = tf32_tr(X - xh), tf32_tr(cent - ch)
    f = lambda a: a.astype(np.float64)                        # noqa: E731
    D = (f(xh) @ f(ch).T + f(xh) @ f(cl).T + f(xl) @ f(ch).T).astype(np.float32)
    scale, bias, A = proxy_terms(cent, metric)
    return (f(D) * f(scale)[None, :] + f(bias)[None, :]).astype(np.float32), A


def old_gate(p0, plast, x, A, metric):
    """The margin this gate replaced: relative to the best proxy, plus 1e-4."""
    return plast < p0 - np.float32(1e-4) * (abs(p0) + np.float32(1))


def new_gate(p0, plast, x, A, metric):
    """assign_shortlist_kernel's gate, in the kernel's fp32 arithmetic."""
    f = np.float32
    d = len(x)
    xn = f(np.sqrt(f((np.asarray(x, np.float64) ** 2).sum()))) * f(1 + 2.0 ** -10)
    gp, gr = f((d + 64) * 2.0 ** -24), f((d // 4 + 24) * 2.0 ** -24)
    if metric == orc.L2:
        e = gp * (xn * A + A * A) + gr * (xn + f(0.5) * A) * (xn + f(0.5) * A)
    elif metric == orc.IP:
        e = (gp + gr) * xn * A
    else:
        e = (gp + f(2) * gr) * xn * A
    return plast < p0 - f(2) * e * f(1 + 2.0 ** -10)


def emulate_shortlist(X, cent, metric, gate, want=None):
    """(accepted, wrong): rows the gate accepts, and accepted rows whose shortlist misses the oracle's winner (the kernel
    would assign another centroid).  A Cosine row below the 1e-6 norm cut is answered 0 without a shortlist."""
    P, A = proxy_scores(X, cent, metric)
    want = oracle_assign(X, cent, metric) if want is None else want
    acc = wrong = 0
    for i in range(len(X)):
        if metric == orc.COSINE and gate is new_gate and orc.norm(X[i]) < 1e-6:
            acc += 1
            wrong += int(want[i] != 0)
            continue
        order = np.argsort(-P[i], kind="stable")[:KPRIME]     # top k', ties to the lower index
        if gate(P[i, order[0]], P[i, order].min(), X[i], A, metric):
            acc += 1
            wrong += int(want[i] not in set(order.tolist()))
    return acc, wrong


def test_emulated_old_gate_accepts_wrong_shortlists():
    """The orthogonal-IP and sphere-L2 regimes defeat the margin relative to the best proxy: most rows are accepted
    with a shortlist that misses the reference's winner."""
    n, nc, d = 200, 2048, 128
    for kind, metric in (("orth_ip_big", orc.IP), ("sphere_l2", orc.L2)):
        X, cent = assign_data(kind, n, nc, d, 11)
        acc, wrong = emulate_shortlist(X, cent, metric, old_gate)
        assert wrong >= n // 2, f"{kind}: old gate accepted {acc}, wrong {wrong} of {n}"


@pytest.mark.parametrize("kind", REGIMES)
def test_emulated_gate_never_accepts_a_shortlist_missing_the_winner(kind):
    n, nc, d = 200, 2048, 128
    X, cent = assign_data(kind, n, nc, d, 12)
    for name, metric in METRICS.items():
        acc, wrong = emulate_shortlist(X, cent, metric, new_gate)
        assert wrong == 0, f"{kind} {name}: {wrong} of {acc} accepted rows miss the oracle's winner"


@pytest.mark.parametrize("kind", ["uniform", "zero_mean"])
def test_emulated_gate_keeps_most_rows(kind):
    """Redoing every row exhaustively would pass the test above: ordinary data must stay on the shortlist."""
    n, nc, d = 400, 2048, 128
    X, cent = assign_data(kind, n, nc, d, 13)
    for name, metric in METRICS.items():
        acc, wrong = emulate_shortlist(X, cent, metric, new_gate)
        assert wrong == 0 and acc >= 0.95 * n, f"{kind} {name}: accepted {acc} of {n}, wrong {wrong}"


def test_emulation_matches_the_oracle_on_exact_data():
    """Sanity of the emulator: small integers are exact in tf32, so the proxy is the exact score and the top proxy
    is the oracle's winner (ties to the lower index)."""
    rng = np.random.default_rng(14)
    X = rng.integers(-8, 9, (64, 16)).astype(np.float32)
    cent = rng.integers(-8, 9, (300, 16)).astype(np.float32)
    for metric in (orc.L2, orc.IP):
        P, _ = proxy_scores(X, cent, metric)
        np.testing.assert_array_equal(np.argmax(P, axis=1), oracle_assign(X, cent, metric))


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    import pyrope_b200 as pg
    pg._lib.check(pg.load().pyrope_gpu_init(0))
    return pg


def _gpu_assign_both_paths(pg, X, cent, metric, monkeypatch):
    a = pg.coarse_assign(X, cent, metric)                    # shortlist at nc >= 2,048 and d % 4 == 0, else exhaustive
    monkeypatch.setenv("PYROPE_ASSIGN_EXACT", "1")
    b = pg.coarse_assign(X, cent, metric)                    # exhaustive exact kernel
    monkeypatch.delenv("PYROPE_ASSIGN_EXACT")
    return a, b


def _assert_rows_equal(got, want, ctx):
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, f"{ctx}: {len(bad)} of {len(want)} rows assigned to another list, e.g. rows {bad[:5].tolist()}: " \
                          f"{got[bad[:5]].tolist()} != oracle {want[bad[:5]].tolist()}"


SHORTLIST_DIMS = [8, 12, 36, 128, 768]
EXHAUSTIVE_DIMS = [1, 3, 7, 130]                             # flat_tc_supported rejects them; 8-lane remainders


@pytest.mark.gpu
@pytest.mark.parametrize("d", SHORTLIST_DIMS + EXHAUSTIVE_DIMS)
@pytest.mark.parametrize("metric", list(METRICS), ids=list(METRICS))
@pytest.mark.parametrize("kind", REGIMES)
def test_coarse_assign_matches_oracle(gpu, monkeypatch, kind, metric, d):
    """Both paths equal the oracle row for row at nc = 2,047 (exhaustive), 2,048 (shortlist) and 5,000."""
    m = METRICS[metric]
    n = 160
    for nc in (2047, 2048, 5000):
        X, cent = assign_data(kind, n, nc, d, 100 + d + nc)
        want = oracle_assign(X, cent, m)
        a, b = _gpu_assign_both_paths(gpu, X, cent, m, monkeypatch)
        _assert_rows_equal(a, want, f"{kind} {metric} d={d} nc={nc} default path")
        _assert_rows_equal(b, want, f"{kind} {metric} d={d} nc={nc} PYROPE_ASSIGN_EXACT")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,metric", [("zero_mean", "L2"), ("orth_ip_big", "IP"), ("zeros", "COSINE")])
def test_coarse_assign_across_the_row_chunk_edge(gpu, monkeypatch, kind, metric):
    """assign_rows shortlists 2^20 rows at a time: rows on both sides of the edge and the last row."""
    m, n, nc, d = METRICS[metric], (1 << 20) + 3000, 2048, 32
    X, cent = assign_data(kind, n, nc, d, 21)
    a, b = _gpu_assign_both_paths(gpu, X, cent, m, monkeypatch)
    rng = np.random.default_rng(22)
    edge = 1 << 20
    sample = np.unique(np.concatenate([np.arange(edge - 200, edge + 200), np.arange(n - 50, n),
                                       rng.choice(n, 300, replace=False)]))
    want = oracle_assign(X[sample], cent, m)
    _assert_rows_equal(a[sample], want, f"{kind} {metric} chunk edge, default path")
    _assert_rows_equal(b[sample], want, f"{kind} {metric} chunk edge, PYROPE_ASSIGN_EXACT")
    _assert_rows_equal(a, b, f"{kind} {metric} all rows, default vs exhaustive")


def _kmeans_data(kind, n, d, seed):
    rng = np.random.default_rng(seed)
    if kind == "orth_ip":                                    # two groups in orthogonal subspaces, 10 and 1e3 long
        X, cent = _orth(n // 2, n - n // 2, d, 10.0, rng, cent_scale=1e3)
        return np.ascontiguousarray(rng.permutation(np.concatenate([X, cent])))
    if kind == "dup":                                        # 24 distinct rows: empty clusters, coinciding centroids
        U = rng.standard_normal((24, d)).astype(np.float32)
        return np.ascontiguousarray(U[rng.integers(0, 24, n)])
    return np.ascontiguousarray(make_data(kind, n, d, 1, seed)[0])


def _assert_kmeans_equal(pg, X, k, metric, iters, ctx):
    gc, git = pg.kmeans_train(X, k, metric, iters, 42)
    rc, rit = orc.kmeans_train(X, k, metric, iters, 42)
    assert gc.shape == rc.shape, f"{ctx}: {gc.shape} != {rc.shape}"
    assert git == rit, f"{ctx}: {git} iterations != oracle {rit}"
    bad = np.flatnonzero((gc != rc).any(1))
    assert len(bad) == 0, f"{ctx}: {len(bad)} of {k} centroids differ, e.g. {bad[:5].tolist()}"


@pytest.mark.gpu
@pytest.mark.parametrize("metric", list(METRICS), ids=list(METRICS))
@pytest.mark.parametrize("kind", ["zero_mean", "mixed", "orth_ip"])
def test_kmeans_shortlist_matches_oracle(gpu, kind, metric):
    """nc = 2,048 takes the shortlist in every iteration; one row assigned elsewhere moves every centroid after it."""
    X = _kmeans_data(kind, 8192, 32, 31)
    _assert_kmeans_equal(gpu, X, 2048, METRICS[metric], 5, f"{kind} {metric}")


@pytest.mark.gpu
@pytest.mark.parametrize("metric", list(METRICS), ids=list(METRICS))
def test_kmeans_exhaustive_odd_dims_duplicates_and_small_n(gpu, metric):
    m = METRICS[metric]
    for d in (3, 7, 130):
        _assert_kmeans_equal(gpu, _kmeans_data("zero_mean", 3000, d, 40 + d), 100, m, 10, f"{metric} d={d}")
    _assert_kmeans_equal(gpu, _kmeans_data("dup", 3000, 16, 41), 64, m, 10, f"{metric} duplicates")
    X = _kmeans_data("zero_mean", 40, 12, 42)
    _assert_kmeans_equal(gpu, X, 40, m, 10, f"{metric} k = n")
    _assert_kmeans_equal(gpu, X, 60, m, 10, f"{metric} k > n")


def _build_data(kind, n, d, seed):
    return np.ascontiguousarray(make_data(kind, n, d, 1, seed)[0])


def _gpu_list_of(off, rows, n):
    lo = np.full(n, -1, np.int64)
    for c in range(len(off) - 1):
        lo[rows[off[c]:off[c + 1]]] = c
    return lo


@pytest.mark.gpu
@pytest.mark.parametrize("index,kind,metric", [
    ("ivf_flat", "zero_mean", "L2"), ("ivf_flat", "mixed", "IP"), ("ivf_flat", "zero_mean", "COSINE"),
    ("ivf_pq", "zero_mean", "L2"), ("ivf_pq", "mixed", "L2")])
def test_build_nlist_2048_matches_oracle(gpu, index, kind, metric):
    """Build at nlist 2,048 (k-means and the final assignment on the shortlist): centroids, lists in order and, for
    IVF_PQ, codebooks, ksub and codes, all equal to the oracle's Build."""
    m, n, d, nlist = METRICS[metric], 8192, 32, 2048
    X = _build_data(kind, n, d, 51)
    if index == "ivf_flat":
        ref = orc.IvfFlatIndex(d, m, nlist=nlist)
        ix = gpu.GpuIndex(gpu.IVF_FLAT, d, m, nlist=nlist)
    else:
        ref = orc.IvfPqIndex(d, m, m=4, k=256, nlist=nlist)
        ix = gpu.GpuIndex(gpu.IVF_PQ, d, m, nlist=nlist, m=4, k=256)
    ref.add_batch(X)
    ref.build()
    ix.add(X)
    ix.build()
    np.testing.assert_array_equal(ix.centroids(), ref.centroids(), err_msg=f"{index} {kind} {metric}: centroids")
    off, rows, codes = ix.lists()
    rl = ref.lists()
    if index == "ivf_pq":
        cb, ks = ix.codebooks()
        np.testing.assert_array_equal(cb, ref.pq().codebook())
        np.testing.assert_array_equal(ks, ref.pq().ksub())
        rl, rcodes = [ids for ids, _ in rl], [c for _, c in rl]
    np.testing.assert_array_equal(np.diff(off), [len(ids) for ids in rl], err_msg="list sizes")
    np.testing.assert_array_equal(rows, np.concatenate(rl), err_msg="list members and order")
    if index == "ivf_pq":
        np.testing.assert_array_equal(codes, np.concatenate(rcodes), err_msg="codes")


@pytest.mark.gpu
def test_extend_orthogonal_ip_rows_land_in_the_oracles_lists(gpu):
    """Extend assigns appended rows with assign_rows (as Build): rows orthogonal to every centroid, |x||c| ~ 1e4 .. 1e5."""
    n0, n1, nlist, d = 3000, 3000, 2048, 32
    X, cent = assign_data("orth_ip_big", n0 + n1, nlist, d, 61)
    ix = gpu.GpuIndex(gpu.IVF_FLAT, d, gpu.INNER_PRODUCT, nlist=nlist)
    ix.set_codebooks(cent)
    ix.add(X[:n0])
    ix.build()
    assert ix.add(X[n0:]) == n0
    ix.extend()
    off, rows, _ = ix.lists()
    got = _gpu_list_of(off, rows, n0 + n1)
    want = oracle_assign(X, cent, orc.IP)
    _assert_rows_equal(got[n0:], want[n0:], "extended rows")
    _assert_rows_equal(got[:n0], want[:n0], "built rows")


SUBS = [1, 2, 3, 4, 5, 6, 7, 8, 15, 16, 17, 31, 32, 33, 48, 64]


@pytest.mark.gpu
@pytest.mark.parametrize("sub", SUBS)
def test_pq_encode_matches_oracle(gpu, sub):
    """ProductQuantizer.Encode (L2SquaredUnsafe, strict '<': lowest code wins): zero-mean residuals, duplicate
    codewords, and ksub < K with the padded codewords set to the rows themselves (they must never be chosen)."""
    rng = np.random.default_rng(70 + sub)
    m, K, n = 3, 256, 400
    cb = rng.standard_normal((m, K, sub)).astype(np.float32)
    cb[0, 200:] = cb[0, 17]                                  # duplicates of codeword 17, and of 5 further down
    cb[1, 9] = cb[1, 250]
    ksub = np.array([K, 100, 7], np.int32)
    X = rng.standard_normal((n, m * sub)).astype(np.float32)
    X[:50, :sub] = cb[0, 17] + 1e-3 * rng.standard_normal((50, sub)).astype(np.float32)
    X[50:60, :sub] = cb[0, 17]
    X[60:70, sub:2 * sub] = cb[1, 9]
    for mi in (1, 2):
        cb[mi, ksub[mi]:] = X[rng.integers(0, n, K - ksub[mi]), mi * sub:(mi + 1) * sub]
    pq = orc.ProductQuantizer(m * sub, m, K)
    pq.set_codebook(cb, ksub)
    want = np.stack([pq.encode(x) for x in X])
    got = gpu.pq_encode(cb, X, ksub)
    for mi in range(m):
        _assert_rows_equal(got[:, mi], want[:, mi], f"sub={sub} subspace {mi}")
    assert (got[:, 1] < 100).all() and (got[:, 2] < 7).all()
    assert (got[50:60, 0] == 17).all()                        # the lowest of the exact duplicates


@pytest.mark.gpu
def test_pq_encode_of_build_residuals_matches_oracle(gpu):
    """Zero-mean residuals of a Build-like assignment against a trained codebook, every sub-vector length of d = 48."""
    rng = np.random.default_rng(80)
    X = rng.standard_normal((3000, 48)).astype(np.float32)
    cent = X[:64].copy()
    R = (X - cent[oracle_assign(X, cent, orc.L2)]).astype(np.float32)
    for m in (48, 24, 16, 12, 8, 6, 4, 3, 2, 1):
        pq = orc.ProductQuantizer(48, m, 64)
        pq.train(R[:1000])
        cb, ks = pq.codebook(), np.array(pq.ksub(), np.int32)
        want = np.stack([pq.encode(r) for r in R])
        _assert_rows_equal(gpu.pq_encode(cb, R, ks).ravel(), want.ravel(), f"m={m}")
