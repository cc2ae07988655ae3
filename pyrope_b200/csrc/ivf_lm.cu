// ivf_lm.cu — K4 list-major IVF_FLAT inverted-list scan (batched).
//
// Replaces IvfFlatVectorIndex.Search:200-218 for a whole query batch.  The reference (and the query-major
// kernel in ivf.cu) streams a probed list once per (query, probe); a batch of 10^4 queries x 16 probes over
// 4096 lists reads every list ~40 times.  Here (query, probe) pairs are grouped BY LIST (counting sort on
// device, same scheme as pq_lm.cu) and one work item is one inverted list x up to 16 of the queries that
// probe it, so a row fetched from L2/HBM is scored against 16 queries.
//
//   ivf_lm_seed_kernel   per query, a lower bound of its k-th best score from a sample of its nearest list, less the
//                        slack two summation orders can differ by (fl_gamma), so no item starts without a threshold;
//   ivf_lm_scan_kernel   persistent CTAs, static item striding, 8 warps.  Lane l holds dimensions 4l..4l+3 of
//                        the item's 16 queries in registers (packed pairs for FFMA2/FADD2); a warp takes two
//                        rows at a time (one coalesced 128-bit load per lane and row, prefetched), forms the
//                        2 x 16 partial scores, and a butterfly reduce-scatter (31 shuffles for 32 sums)
//                        leaves lane l with the complete score of (row l/16, query l%16), which it tests
//                        against that query's threshold.  Candidates go to a per-slot queue; after the item
//                        one warp per slot hands at most k of them to the pair's private pool region and
//                        tightens the query's threshold (atomicMax);
//   ivf_lm_redo_kernel   plain scan, in the reference's order, of a (query, list) whose queue overflowed or whose
//                        best k could not be told from the rest within the slack;
//   ivf_lm_final_kernel  every pool entry within the slack of the k-th, RE-SCORED in the reference's evaluation order
//                        (VectorMath.L2Squared / DotProduct, VectorMath.cs:8-70), the best k of them reported: the
//                        oracle's rows and scores bit for bit.
// Shapes: L2 / inner product / cosine, dim % 4 == 0 and dim <= 1024 (rows wider than 128 floats take the *_wide kernels),
// no MaxScans budget; everything else takes ivf.cu.
#include <cub/cub.cuh>

#include <cstdio>

#include "common.cuh"
#include "exact_arith.cuh"
#include "kernels.h"

namespace pyrope {
namespace {

constexpr int FG = 16;         // queries per work item
constexpr int FT = 256;        // threads (8 warps)
constexpr int FQC = 256;       // candidate queue entries per slot
constexpr int FSEED = 512;     // rows sampled per query for the starting threshold
constexpr int FREDO_QCAP = 2048;

__device__ __forceinline__ unsigned long long pack2(float a, float b) {
    unsigned long long d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(a), "f"(b));
    return d;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& a, float& b) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ unsigned long long fadd2(unsigned long long a, unsigned long long b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// ---- grouping ----------------------------------------------------------------------------------------
__global__ void fl_count_kernel(const int64_t* __restrict__ probes, int64_t npairs, const int64_t* __restrict__ list_off,
                                int32_t* lcnt, unsigned long long* scanned) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long len = 0;
    if (i < npairs) {
        const int64_t l = probes[i];
        if (l >= 0) {
            len = (unsigned long long)(list_off[l + 1] - list_off[l]);
            if (len) atomicAdd(&lcnt[l], 1);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) len += __shfl_xor_sync(0xffffffffu, len, o);
    if ((threadIdx.x & 31) == 0 && len) atomicAdd(scanned, len);
}
__global__ void fl_items_per_list_kernel(const int32_t* __restrict__ lcnt, int nlist, int32_t* nit) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= nlist) nit[i] = i < nlist ? (lcnt[i] + FG - 1) / FG : 0;
}
__global__ void fl_fill_pairs_kernel(const int64_t* __restrict__ probes, int64_t npairs, int P,
                                     const int64_t* __restrict__ list_off, const int32_t* __restrict__ loff, int32_t* lcur,
                                     int32_t* pairq, int32_t* pairp) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npairs) return;
    const int64_t l = probes[i];
    if (l >= 0 && list_off[l + 1] > list_off[l]) {
        const int slot = loff[l] + atomicAdd(&lcur[l], 1);
        pairq[slot] = (int32_t)(i / P);
        pairp[slot] = (int32_t)(i % P);
    }
}
__global__ void fl_fill_items_kernel(const int32_t* __restrict__ nit, const int32_t* __restrict__ ioff, int nlist, int2* items) {
    int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= nlist) return;
    const int n = nit[l], o = ioff[l];
    for (int g = 0; g < n; ++g) items[o + g] = make_int2(l, g);
}

// score of one row against one query, plain fp32 (one warp, lane = 4 dims); L2 -> -|q-x|^2, IP -> q.x
template <int METRIC>
__device__ __forceinline__ float warp_score(const float4 qv, const float4 xv) {
    float a;
    if (METRIC == kL2) {
        const float d0 = qv.x - xv.x, d1 = qv.y - xv.y, d2 = qv.z - xv.z, d3 = qv.w - xv.w;
        a = -(fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, d3 * d3))));
    } else {  // inner product; Cosine callers scale by 1 / |x| (inv_norm)
        a = fmaf(qv.x, xv.x, fmaf(qv.y, xv.y, fmaf(qv.z, xv.z, qv.w * xv.w)));
    }
    return warp_sum(a);
}

// Cosine ranks a query's rows by q.x / |x| (its own norm is a positive constant): the proxy every kernel below compares and
// queues; the final kernel re-scores with VectorMath.Cosine's guards (0 below 1e-6, VectorMath.cs:102-109).
__device__ __forceinline__ float inv_norm(const float* __restrict__ norms, int64_t pos) {
    const float n = __ldg(norms + pos);
    return n < 1e-6f ? 0.f : 1.f / n;
}

// The seed, the scan, the redo and VectorMath (the reference) sum a row's products in different orders.  Each order is
// within gamma_n sum|term| of the exact sum, n its depth: d/8 + 8 for the reference, at most d/32 + 9 here; two of them
// differ by at most fl_gamma(d) sum|term| (the slack also covers the 1 / (1 - n u) factors and Cosine's scaling).  L2's
// terms are non-negative, so sum|term| is the score's magnitude; for IP and the Cosine proxy it is not bounded by the
// score at all (rows orthogonal to the query score rounding noise), and the seed bounds it (FlSeed::band).
__host__ __device__ __forceinline__ float fl_gamma(int dim) { return (float)(dim / 4 + 24) * 0x1p-24f; }
// how far below a score t another order can put a row that ranks with t in the reference's order, twice over (the row's
// own error and the error of the row that set t): band = fl_gamma * max sum|term| (0 for L2)
__device__ __forceinline__ float fl_slack(float t, float band, float gam) { return 2.f * (band + gam * fabsf(t)) + 1e-30f; }

__device__ __forceinline__ float warp_abs(const float4 qv, const float4 xv) {
    return warp_sum(fmaf(fabsf(qv.x), fabsf(xv.x), fmaf(fabsf(qv.y), fabsf(xv.y), fmaf(fabsf(qv.z), fabsf(xv.z), fabsf(qv.w * xv.w)))));
}

// ---- seed: a lower bound of every query's k-th best score -------------------------------------------------
struct FlSeed {
    const float* Q; int64_t nq; int dim; const int64_t* probes; int P;
    const float* vecs; const uint8_t* dead; const int64_t* list_off;
    uint32_t* pool_thr; int k;
    const float* norms;  // Cosine: |x| per list entry
    float* band;         // per query, fl_gamma times a bound of sum|q_i x_i|: IP, the largest over the rows sampled;
                         // Cosine (the proxy divides by |x|), |q| (Cauchy-Schwarz)
};
template <int METRIC>
__global__ void __launch_bounds__(256) ivf_lm_seed_kernel(FlSeed a) {
    const int64_t q = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (q >= a.nq) return;
    float4 qv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane * 4 < a.dim) qv = __ldg(reinterpret_cast<const float4*>(a.Q + q * a.dim) + lane);
    constexpr int U = FSEED / 32;
    float sc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) sc[u] = -INFINITY;
    int got = 0;
    float amax = 0.f;
    for (int pr = 0; pr < a.P && got < min(max(a.k, 32), FSEED); ++pr) {
        const int64_t l = a.probes[q * a.P + pr];
        if (l < 0) continue;
        const int64_t beg = a.list_off[l], len = a.list_off[l + 1] - beg;
        for (int64_t v0 = 0; v0 < len && got < FSEED; v0 += 8) {  // eight rows in flight per step
            float4 xv[8];
            bool ok[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int64_t v = v0 + u;
                ok[u] = v < len && !(a.dead && a.dead[beg + v]);  // warp-uniform
                xv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok[u] && lane * 4 < a.dim) xv[u] = __ldg(reinterpret_cast<const float4*>(a.vecs + (beg + v) * a.dim) + lane);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                if (ok[u] && got < FSEED) {
                    float s = warp_score<METRIC>(qv, xv[u]);
                    if (METRIC == kCosine) s *= inv_norm(a.norms, beg + v0 + u);
                    if (METRIC == kIP) amax = fmaxf(amax, warp_abs(qv, xv[u]));
#pragma unroll
                    for (int w = 0; w < U; ++w)
                        if ((got >> 5) == w && (got & 31) == lane) sc[w] = s;
                    ++got;
                }
            }
        }
    }
    if (METRIC == kCosine) amax = sqrtf(warp_abs(qv, qv));  // sum|q_i x_i| / |x| <= |q| for every row
    const float gam = fl_gamma(a.dim), band = gam * amax * (1.f + 0x1p-10f);
    if (lane == 0) a.band[q] = band;
    if (got < a.k) return;  // fewer candidates than k so far: no threshold (everything is kept)
    // k-th largest of the sampled scores by bisection on the ordered bits
    uint32_t o[U], lo = 0xffffffffu, hi = 0u;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        o[u] = sc[u] == -INFINITY ? 0u : score_to_ord(sc[u]);
        if (o[u]) { lo = min(lo, o[u]); hi = max(hi, o[u]); }
    }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo + 1u) >> 1);
        int c = 0;
#pragma unroll
        for (int u = 0; u < U; ++u) c += o[u] >= mid;
        c = __reduce_add_sync(0xffffffffu, c);
        if (c >= a.k) lo = mid; else hi = mid - 1u;
    }
    if (lane == 0) {
        // the scan sums the same products in another order, the final ranking in the reference's: leave room for both
        const float t = ord_to_score(lo);
        const float tl = t - fl_slack(t, band, gam);
        a.pool_thr[q] = score_to_ord(tl) - 1u;  // accept iff score >= tl
    }
}

// ---- scan ---------------------------------------------------------------------------------------------------
struct FlParams {
    const float* Q; int dim; const float* vecs; const uint8_t* dead; const int64_t* list_off;
    const int2* items; const int32_t* n_items; const int32_t* pair_off; const int32_t* pairq; const int32_t* pairp;
    unsigned long long* pool; int32_t* pool_cnt; uint32_t* pool_thr; int pslots; int k;
    int2* redo; int32_t* redo_cnt;
    const float* norms;  // Cosine: |x| per list entry
    const float* band;   // FlSeed::band
};

// ---- after an item: hand at most k candidates per slot to the pair's private pool region, tighten the threshold ------
// The pool keeps the best k of a pair by the scan's scores.  When the best one left out is within the slack of the k-th,
// the cut may disagree with the reference's order: the pair goes to the redo kernel, which ranks in that order.  The
// published threshold trails the k-th by the slack, so no row the reference ranks above it is turned away.
template <int METRIC>
__device__ __forceinline__ void fl_hand_over(const FlParams& p, int it, uint64_t* qkeys, int* s_qcnt, const int* s_qid,
                                             const int* s_psl, int warp, int lane, float gam) {
    for (int j = warp; j < FG; j += FT / 32) {
        const int n = s_qcnt[j];
        const int q = s_qid[j];
        if (n > 0 && q >= 0) {
            uint64_t* kq = qkeys + j * FQC;
            if (n > FQC) {
                if (lane == 0) p.redo[atomicAdd(p.redo_cnt, 1)] = make_int2(q, it * FG + j);
            } else {
                const size_t ps = (size_t)q * p.pslots + s_psl[j];
                unsigned long long* dst = p.pool + ps * p.k;
                uint64_t mink = ~0ull, next = 0ull;  // the k-th kept, the best left out
                int kept;
                if (n > p.k && n <= 64) {  // select by rank counting inside the warp
                    const uint64_t a = lane < n ? kq[lane] : 0ull, b = lane + 32 < n ? kq[lane + 32] : 0ull;
                    int ra = 0, rb = 0;
                    for (int i = 0; i < n; ++i) {
                        const uint64_t x = kq[i];
                        ra += x > a;
                        rb += x > b;
                    }
                    const bool ka = lane < n && ra < p.k, kb = lane + 32 < n && rb < p.k;
                    const unsigned ma = __ballot_sync(0xffffffffu, ka), mb = __ballot_sync(0xffffffffu, kb);
                    kept = __popc(ma) + __popc(mb);
                    const unsigned below = (1u << lane) - 1u;
                    if (ka) { dst[__popc(ma & below)] = a; mink = a; }
                    if (kb) { dst[__popc(ma) + __popc(mb & below)] = b; mink = b < mink ? b : mink; }
                    if (lane < n && !ka) next = a;
                    if (lane + 32 < n && !kb) next = b > next ? b : next;
                } else {
                    if (n > p.k) {
                        const int P2 = next_pow2(n);
                        for (int i = n + lane; i < P2; i += 32) kq[i] = 0ull;
                        __syncwarp();
                        bitonic_sort_desc<true>(kq, P2, lane, 32);
                    }
                    kept = min(n, p.k);
                    for (int i = lane; i < kept; i += 32) {
                        const uint64_t x = kq[i];
                        dst[i] = x;
                        mink = x < mink ? x : mink;
                    }
                    if (n > p.k) next = kq[p.k];
                }
                if (lane == 0) p.pool_cnt[ps] = kept;
                if (kept >= p.k) {
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const uint64_t x = __shfl_xor_sync(0xffffffffu, mink, o), y = __shfl_xor_sync(0xffffffffu, next, o);
                        mink = x < mink ? x : mink;
                        next = y > next ? y : next;
                    }
                    if (lane == 0) {
                        const float m = key_score(mink), band = p.band[q];
                        const float lim = m - fl_slack(m, band, gam);
                        atomicMax(p.pool_thr + q, score_to_ord(lim) - 1u);
                        // L2's slack is relative: a cut inside it is a tie within 2 fl_gamma of the score
                        if (METRIC != kL2 && next && key_score(next) >= lim) p.redo[atomicAdd(p.redo_cnt, 1)] = make_int2(q, it * FG + j);
                    }
                }
            }
        }
        __syncwarp();
        if (lane == 0) s_qcnt[j] = 0;
    }
}

template <int METRIC>
__global__ void __launch_bounds__(FT, 2) ivf_lm_scan_kernel(FlParams p) {
    __shared__ uint64_t qkeys[FG * FQC];
    __shared__ int s_qcnt[FG];
    __shared__ int s_qid[FG], s_psl[FG];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_items = *p.n_items;
    const int dim = p.dim;
    const bool lane_on = lane * 4 < dim;
    const float gam = fl_gamma(dim);
    if (tid < FG) s_qcnt[tid] = 0;
    __syncthreads();

    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
        const int2 item = __ldg(&p.items[it]);
        const int l = item.x, g = item.y;
        const int64_t beg = __ldg(p.list_off + l), len = __ldg(p.list_off + l + 1) - beg;
        const int pbeg = __ldg(p.pair_off + l), pend = __ldg(p.pair_off + l + 1);
        if (tid < FG) {
            const int idx = pbeg + FG * g + tid;
            s_qid[tid] = idx < pend ? __ldg(p.pairq + idx) : -1;
            s_psl[tid] = idx < pend ? __ldg(p.pairp + idx) : 0;
        }
        __syncthreads();
        // this lane's 4 dimensions of the 16 queries, packed in pairs (query 2j, 2j+1) for the f32x2 pipes
        unsigned long long qp[FG / 2][4];
#pragma unroll
        for (int j = 0; j < FG / 2; ++j) {
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
            const int qa = s_qid[2 * j], qb = s_qid[2 * j + 1];
            if (lane_on && qa >= 0) a = __ldg(reinterpret_cast<const float4*>(p.Q + (size_t)qa * dim) + lane);
            if (lane_on && qb >= 0) b = __ldg(reinterpret_cast<const float4*>(p.Q + (size_t)qb * dim) + lane);
            qp[j][0] = pack2(a.x, b.x); qp[j][1] = pack2(a.y, b.y); qp[j][2] = pack2(a.z, b.z); qp[j][3] = pack2(a.w, b.w);
        }
        // after the reduce-scatter lane holds (row = lane / 16, query = lane % 16)
        const int myq = s_qid[lane & 15];
        float thr = INFINITY;  // nothing passes for an empty slot
        if (myq >= 0) {
            const uint32_t u = __ldcg(p.pool_thr + myq);
            thr = u ? ord_to_score(u) : -INFINITY;
        }

        const float4* rows = reinterpret_cast<const float4*>(p.vecs + (size_t)beg * dim);
        const int rstride = dim / 4;
        const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
        int64_t v = 2 * warp;
        float4 n0 = zero4, n1 = zero4;
        if (lane_on && v < len) n0 = __ldg(rows + v * rstride + lane);
        if (lane_on && v + 1 < len) n1 = __ldg(rows + (v + 1) * rstride + lane);
        for (; v < len; v += 2 * (FT / 32)) {
            const float4 x0 = n0, x1 = n1;
            const int64_t vn = v + 2 * (FT / 32);
            if (lane_on && vn < len) n0 = __ldg(rows + vn * rstride + lane);
            if (lane_on && vn + 1 < len) n1 = __ldg(rows + (vn + 1) * rstride + lane);
            float vals[32];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const float4 x = r ? x1 : x0;
                const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int j = 0; j < FG / 2; ++j) {
                    unsigned long long acc = 0ull;
#pragma unroll
                    for (int d = 0; d < 4; ++d) {
                        if (METRIC == kL2) {
                            const unsigned long long df = fadd2(qp[j][d], pack2(-xs[d], -xs[d]));
                            acc = ffma2(df, df, acc);
                        } else {
                            acc = ffma2(qp[j][d], pack2(xs[d], xs[d]), acc);
                        }
                    }
                    unpack2(acc, vals[r * 16 + 2 * j], vals[r * 16 + 2 * j + 1]);
                }
            }
            // butterfly reduce-scatter: 32 partial sums x 32 lanes -> lane i holds the total of value i
#pragma unroll
            for (int s = 16; s >= 1; s >>= 1) {
                const bool upper = (lane & s) != 0;
#pragma unroll
                for (int i = 0; i < s; ++i) {
                    const float send = upper ? vals[i] : vals[i + s];
                    const float keep = upper ? vals[i + s] : vals[i];
                    vals[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
                }
            }
            float score = METRIC == kL2 ? -vals[0] : vals[0];
            const int64_t row = v + (lane >> 4);
            if (METRIC == kCosine && row < len) score *= inv_norm(p.norms, beg + row);
            if (row < len && score > thr) {
                const int64_t gpos = beg + row;
                if (!(p.dead && p.dead[gpos])) {
                    const int j = lane & 15;
                    const int pos = atomicAdd(&s_qcnt[j], 1);
                    if (pos < FQC) qkeys[j * FQC + pos] = make_key(score, (uint32_t)gpos);
                }
            }
        }
        __syncthreads();
        fl_hand_over<METRIC>(p, it, qkeys, s_qcnt, s_qid, s_psl, warp, lane, gam);
        __syncthreads();
    }
}

// ---- rows wider than 128 floats (d <= 1024) ---------------------------------------------------------------------
// Same item / pool / threshold scheme; what changes is where the 16 queries live.  A lane cannot hold d/32 dimensions of 16
// queries in registers, so the item's queries are staged in shared memory once, interleaved per 128-dimension chunk, and
// the loop nest is turned inside out: a warp owns a block of 32 rows, walks the chunks, re-loads its query registers
// once per (block, chunk) - 32 LDS.64 for 16 row pairs - and keeps the running (row, query) sums of the block in a
// private strip of shared memory (lane i always touches the same 16 slots: no synchronisation).
constexpr int FW_MAX_DIM = 1024;
constexpr int FWR = 32;      // rows per warp and pass
constexpr int FSEEDW = FSEED;  // rows sampled per query for the starting threshold: as many as for narrow rows - with 64 the
                               // k-th of the sample let 15 % of a list through, most pairs overflowed their queue and the
                               // redo kernel (one CTA per pair) ran for 0.75 s next to a 0.1 s scan

template <int METRIC>
__device__ __forceinline__ float warp_score_wide(const float* __restrict__ q, const float* __restrict__ x, int dim, int lane) {
    float a = 0.f;
    for (int c = lane * 4; c < dim; c += 128) {
        const float4 qv = __ldg(reinterpret_cast<const float4*>(q + c)), xv = __ldg(reinterpret_cast<const float4*>(x + c));
        if (METRIC == kL2) {
            const float d0 = qv.x - xv.x, d1 = qv.y - xv.y, d2 = qv.z - xv.z, d3 = qv.w - xv.w;
            a = fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, fmaf(d3, d3, a))));
        } else {
            a = fmaf(qv.x, xv.x, fmaf(qv.y, xv.y, fmaf(qv.z, xv.z, fmaf(qv.w, xv.w, a))));
        }
    }
    a = warp_sum(a);
    return METRIC == kL2 ? -a : a;
}
__device__ __forceinline__ float warp_abs_wide(const float* __restrict__ q, const float* __restrict__ x, int dim, int lane) {
    float a = 0.f;
    for (int c = lane * 4; c < dim; c += 128) {
        const float4 qv = __ldg(reinterpret_cast<const float4*>(q + c)), xv = __ldg(reinterpret_cast<const float4*>(x + c));
        a = fmaf(fabsf(qv.x), fabsf(xv.x), fmaf(fabsf(qv.y), fabsf(xv.y), fmaf(fabsf(qv.z), fabsf(xv.z), fmaf(fabsf(qv.w), fabsf(xv.w), a))));
    }
    return warp_sum(a);
}

template <int METRIC>
__global__ void __launch_bounds__(256) ivf_lm_seed_wide_kernel(FlSeed a) {
    const int64_t q = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (q >= a.nq) return;
    constexpr int U = FSEEDW / 32;
    float sc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) sc[u] = -INFINITY;
    const int want = FSEEDW;
    int got = 0;
    float amax = 0.f;
    for (int pr = 0; pr < a.P && got < want; ++pr) {
        const int64_t l = a.probes[q * a.P + pr];
        if (l < 0) continue;
        const int64_t beg = a.list_off[l], len = a.list_off[l + 1] - beg;
        for (int64_t v = 0; v < len && got < want; ++v) {
            if (a.dead && a.dead[beg + v]) continue;  // warp-uniform
            float s = warp_score_wide<METRIC>(a.Q + q * a.dim, a.vecs + (beg + v) * a.dim, a.dim, lane);
            if (METRIC == kCosine) s *= inv_norm(a.norms, beg + v);
            if (METRIC == kIP) amax = fmaxf(amax, warp_abs_wide(a.Q + q * a.dim, a.vecs + (beg + v) * a.dim, a.dim, lane));
#pragma unroll
            for (int w = 0; w < U; ++w)
                if ((got >> 5) == w && (got & 31) == lane) sc[w] = s;
            ++got;
        }
    }
    if (METRIC == kCosine) amax = sqrtf(warp_abs_wide(a.Q + q * a.dim, a.Q + q * a.dim, a.dim, lane));  // |q|
    const float gam = fl_gamma(a.dim), band = gam * amax * (1.f + 0x1p-10f);
    if (lane == 0) a.band[q] = band;
    if (got < a.k) return;  // fewer candidates than k so far: no threshold (everything is kept)
    uint32_t o[U], lo = 0xffffffffu, hi = 0u;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        o[u] = sc[u] == -INFINITY ? 0u : score_to_ord(sc[u]);
        if (o[u]) { lo = min(lo, o[u]); hi = max(hi, o[u]); }
    }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    while (lo < hi) {  // k-th largest of the sampled scores
        const uint32_t mid = lo + ((hi - lo + 1u) >> 1);
        int c = 0;
#pragma unroll
        for (int u = 0; u < U; ++u) c += o[u] >= mid;
        c = __reduce_add_sync(0xffffffffu, c);
        if (c >= a.k) lo = mid; else hi = mid - 1u;
    }
    if (lane == 0) {
        const float t = ord_to_score(lo);
        const float tl = t - fl_slack(t, band, gam);  // room for the scan's and the reference's summation orders
        a.pool_thr[q] = score_to_ord(tl) - 1u;
    }
}

template <int METRIC>
__global__ void __launch_bounds__(FT, 2) ivf_lm_scan_wide_kernel(FlParams p, int nchunk) {
    extern __shared__ __align__(16) unsigned char fw_smem[];
    float2* s_q2 = reinterpret_cast<float2*>(fw_smem);                        // [nchunk][8 query pairs][4 dims][32 lanes]
    float* s_part = reinterpret_cast<float*>(s_q2 + (size_t)nchunk * 1024);   // [8 warps][FWR rows x 16 queries]
    __shared__ uint64_t qkeys[FG * FQC];
    __shared__ int s_qcnt[FG];
    __shared__ int s_qid[FG], s_psl[FG];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_items = *p.n_items;
    const int dim = p.dim;
    const float gam = fl_gamma(dim);
    if (tid < FG) s_qcnt[tid] = 0;
    __syncthreads();

    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
        const int2 item = __ldg(&p.items[it]);
        const int l = item.x, g = item.y;
        const int64_t beg = __ldg(p.list_off + l), len = __ldg(p.list_off + l + 1) - beg;
        const int pbeg = __ldg(p.pair_off + l), pend = __ldg(p.pair_off + l + 1);
        if (tid < FG) {
            const int idx = pbeg + FG * g + tid;
            s_qid[tid] = idx < pend ? __ldg(p.pairq + idx) : -1;
            s_psl[tid] = idx < pend ? __ldg(p.pairp + idx) : 0;
        }
        __syncthreads();
        // the item's queries, pair (2j, 2j+1) interleaved: entry ((c*8 + j)*4 + d)*32 + lane = dimension c*128 + lane*4 + d
        for (int i = tid; i < nchunk * 1024; i += FT) {
            const int ln = i & 31, d = (i >> 5) & 3, j = (i >> 7) & 7, c = i >> 10;
            const int dd = c * 128 + ln * 4 + d;
            const int qa = s_qid[2 * j], qb = s_qid[2 * j + 1];
            float a = 0.f, b = 0.f;
            if (dd < dim) {
                if (qa >= 0) a = __ldg(p.Q + (size_t)qa * dim + dd);
                if (qb >= 0) b = __ldg(p.Q + (size_t)qb * dim + dd);
            }
            s_q2[i] = make_float2(a, b);
        }
        __syncthreads();
        const int myq = s_qid[lane & 15];  // after the reduce-scatter a lane holds (row = lane / 16, query = lane % 16)
        float thr = INFINITY;              // nothing passes for an empty slot
        if (myq >= 0) {
            const uint32_t u = __ldcg(p.pool_thr + myq);
            thr = u ? ord_to_score(u) : -INFINITY;
        }
        const float4* rows = reinterpret_cast<const float4*>(p.vecs + (size_t)beg * dim);
        const int rstride = dim / 4;
        const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
        float* part = s_part + warp * (FWR * 16);
        for (int64_t rb = (int64_t)warp * FWR; rb < len; rb += (int64_t)(FT / 32) * FWR) {
            const int npair = (int)min((int64_t)(FWR / 2), (len - rb + 1) / 2);
            for (int c = 0; c < nchunk; ++c) {
                unsigned long long qp[FG / 2][4];
#pragma unroll
                for (int j = 0; j < FG / 2; ++j)
#pragma unroll
                    for (int d = 0; d < 4; ++d)
                        qp[j][d] = *reinterpret_cast<const unsigned long long*>(&s_q2[((c * 8 + j) * 4 + d) * 32 + lane]);
                const bool lane_on = c * 128 + lane * 4 < dim;
                const float4* rc = rows + c * 32 + lane;
                float4 n0 = zero4, n1 = zero4;
                if (lane_on) n0 = __ldg(rc + rb * rstride);
                if (lane_on && rb + 1 < len) n1 = __ldg(rc + (rb + 1) * rstride);
#pragma unroll 1
                for (int rp = 0; rp < npair; ++rp) {
                    const float4 x0 = n0, x1 = n1;
                    const int64_t vn = rb + 2 * (rp + 1);
                    n0 = zero4; n1 = zero4;
                    if (lane_on && rp + 1 < npair) n0 = __ldg(rc + vn * rstride);
                    if (lane_on && rp + 1 < npair && vn + 1 < len) n1 = __ldg(rc + (vn + 1) * rstride);
                    float vals[32];
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        const float4 x = r ? x1 : x0;
                        const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                        for (int j = 0; j < FG / 2; ++j) {
                            unsigned long long acc = 0ull;
#pragma unroll
                            for (int d = 0; d < 4; ++d) {
                                if (METRIC == kL2) {
                                    const unsigned long long df = fadd2(qp[j][d], pack2(-xs[d], -xs[d]));
                                    acc = ffma2(df, df, acc);
                                } else {
                                    acc = ffma2(qp[j][d], pack2(xs[d], xs[d]), acc);
                                }
                            }
                            unpack2(acc, vals[r * 16 + 2 * j], vals[r * 16 + 2 * j + 1]);
                        }
                    }
#pragma unroll
                    for (int s2 = 16; s2 >= 1; s2 >>= 1) {  // butterfly reduce-scatter: lane i ends with the total of value i
                        const bool upper = (lane & s2) != 0;
#pragma unroll
                        for (int i = 0; i < s2; ++i) {
                            const float send = upper ? vals[i] : vals[i + s2];
                            const float keep = upper ? vals[i + s2] : vals[i];
                            vals[i] = keep + __shfl_xor_sync(0xffffffffu, send, s2);
                        }
                    }
                    float* ps = part + rp * 32 + lane;  // (row 2 rp + lane / 16, query lane % 16)
                    *ps = c == 0 ? vals[0] : *ps + vals[0];
                }
            }
            for (int rp = 0; rp < npair; ++rp) {
                const int64_t row = rb + 2 * rp + (lane >> 4);
                float score = part[rp * 32 + lane];
                if (METRIC == kL2) score = -score;
                if (METRIC == kCosine && row < len) score *= inv_norm(p.norms, beg + row);
                if (row < len && score > thr) {
                    const int64_t gpos = beg + row;
                    if (!(p.dead && p.dead[gpos])) {
                        const int j = lane & 15;
                        const int pos = atomicAdd(&s_qcnt[j], 1);
                        if (pos < FQC) qkeys[j * FQC + pos] = make_key(score, (uint32_t)gpos);
                    }
                }
            }
        }
        __syncthreads();
        fl_hand_over<METRIC>(p, it, qkeys, s_qcnt, s_qid, s_psl, warp, lane, gam);
        __syncthreads();
    }
}

// ---- redo: plain scan of one (query, list) whose queue overflowed or whose cut fell inside the slack -------------
// IP / Cosine: one thread per row, in the reference's summation order, so the best k it keeps are the reference's (the
// Cosine proxy divides by the row's norm as the scan does).  L2: one warp per row in the scan's order.
struct FlRedo {
    const float* Q; int dim; const float* vecs; const uint8_t* dead; const int64_t* list_off;
    const int2* items; const int32_t* pair_off; const int32_t* pairp;
    const int2* redo; const int32_t* redo_cnt;
    unsigned long long* pool; int32_t* pool_cnt; int pslots; int k;
    const uint32_t* pool_thr;  // the query's current threshold: a valid bound, so the redo queue starts warm
    const float* norms;
};
template <int METRIC>
__global__ void __launch_bounds__(256) ivf_lm_redo_kernel(FlRedo a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem_raw);  // [FREDO_QCAP]
    float* qs = reinterpret_cast<float*>(keys + FREDO_QCAP);  // [dim]
    __shared__ int s_cnt;
    __shared__ uint64_t s_thr;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_redo = *a.redo_cnt;
    for (int e = blockIdx.x; e < n_redo; e += gridDim.x) {
        const int2 en = a.redo[e];
        const int2 item = a.items[en.y / FG];
        const int l = item.x;
        const int64_t beg = a.list_off[l], len = a.list_off[l + 1] - beg;
        const size_t ps = (size_t)en.x * a.pslots + a.pairp[a.pair_off[l] + FG * item.y + en.y % FG];
        __syncthreads();
        CtaQueue Qu{keys, &s_cnt, &s_thr, FREDO_QCAP, a.k};
        Qu.reset(tid);
        __syncthreads();
        if (tid == 0) s_thr = (uint64_t)__ldcg(a.pool_thr + en.x) << 32;  // keys at or below it cannot be in the top k
        for (int d = tid; d < a.dim; d += 256) qs[d] = a.Q[(size_t)en.x * a.dim + d];
        __syncthreads();
        for (int64_t c0 = 0; c0 < len; c0 += 256) {
            if (s_cnt + 256 > FREDO_QCAP) Qu.prune(tid, 256);
            if (METRIC == kL2) {
                const bool wide = a.dim > 128;
                float4 qv = make_float4(0.f, 0.f, 0.f, 0.f);
                if (!wide && lane * 4 < a.dim) qv = reinterpret_cast<const float4*>(qs)[lane];
                for (int64_t v = c0 + warp; v < min(len, c0 + 256); v += 8) {
                    float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (!wide && lane * 4 < a.dim) xv = __ldg(reinterpret_cast<const float4*>(a.vecs + (beg + v) * a.dim) + lane);
                    const float s = wide ? warp_score_wide<kL2>(a.Q + (size_t)en.x * a.dim, a.vecs + (beg + v) * a.dim, a.dim, lane)
                                         : warp_score<kL2>(qv, xv);
                    if (lane == 0 && !(a.dead && a.dead[beg + v])) Qu.push(make_key(s, (uint32_t)(beg + v)));
                }
                __syncthreads();
                continue;
            }
            const int64_t v = c0 + tid;
            if (v < len && !(a.dead && a.dead[beg + v])) {
                const float* x = a.vecs + (beg + v) * a.dim;
                float s = METRIC == kL2 ? -exact::a2_eval<0>(qs, x, a.dim) : exact::a2_eval<1>(qs, x, a.dim);
                if (METRIC == kCosine) s *= inv_norm(a.norms, beg + v);
                Qu.push(make_key(s, (uint32_t)(beg + v)));
            }
            __syncthreads();
        }
        Qu.prune(tid, 256);
        const int keep = s_cnt;
        if (tid == 0) a.pool_cnt[ps] = keep;
        for (int i = tid; i < keep; i += 256) a.pool[ps * a.k + i] = keys[i];
    }
}

// ---- pool -> best k in the reference's order, final order ----------------------------------------------------
// The pool's keys hold the scan's scores.  Every entry within the slack of the k-th of them is re-scored in the
// reference's order (no entry below can reach the reference's k-th), and the best k of those are reported.
struct FlFinal {
    const float* Q; int dim; const float* vecs; const int64_t* labels;
    const unsigned long long* pool; const int32_t* pool_cnt; int pslots; int k; int metric;
    const float* norms; const float* qnorm;  // Cosine
    const float* band;                       // FlSeed::band
    PairOut out;
};
__global__ void __launch_bounds__(256) ivf_lm_final_kernel(FlFinal p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem_raw);
    float* qs = reinterpret_cast<float*>(keys + next_pow2(max(2, p.pslots * p.k)));  // [dim]
    const int64_t q = blockIdx.x;
    const int tid = threadIdx.x;
    __shared__ int s_n;
    if (tid == 0) s_n = 0;
    for (int d = tid; d < p.dim; d += blockDim.x) qs[d] = p.Q[q * p.dim + d];
    __syncthreads();
    for (int sl = tid; sl < p.pslots; sl += blockDim.x) {
        const size_t ps = (size_t)q * p.pslots + sl;
        const int c = min(p.pool_cnt[ps], p.k);
        if (c > 0) {
            const int base = atomicAdd(&s_n, c);
            for (int i = 0; i < c; ++i) keys[base + i] = p.pool[ps * p.k + i];
        }
    }
    __shared__ int s_nr;
    if (tid == 0) s_nr = 0;
    __syncthreads();
    const int n = s_n;
    const int kk = min(n, p.k);
    int nr = n;  // entries to re-score
    if (n > kk) {
        const int P2 = next_pow2(max(n, 2));
        for (int i = n + tid; i < P2; i += blockDim.x) keys[i] = 0ull;
        __syncthreads();
        bitonic_sort_desc<false>(keys, P2, tid, blockDim.x);
        const float m = key_score(keys[kk - 1]);
        const float lim = m - fl_slack(m, p.band[q], fl_gamma(p.dim));
        int c = 0;
        for (int i = kk + tid; i < n; i += blockDim.x) c += key_score(keys[i]) >= lim;
        if (c) atomicAdd(&s_nr, c);
        __syncthreads();
        nr = kk + s_nr;
    }
    __syncthreads();
    // IvfFlatVectorIndex.ComputeScore (:351-360): -L2Squared / DotProduct in VectorMath's single-accumulator order
    for (int i = tid; i < nr; i += blockDim.x) {
        const uint32_t pos = key_pos(keys[i]);
        const float* x = p.vecs + (size_t)pos * p.dim;
        float s = p.metric == kL2 ? -exact::a2_eval<0>(qs, x, p.dim) : exact::a2_eval<1>(qs, x, p.dim);
        if (p.metric == kCosine) {  // VectorMath.Cosine (VectorMath.cs:102-109) on the stored norms
            const float qn = p.qnorm[q], xn = p.norms[pos];
            s = (qn < 1e-6f || xn < 1e-6f) ? 0.f : __fdiv_rn(s, __fmul_rn(qn, xn));
        }
        keys[i] = make_key(s, pos);
    }
    __syncthreads();
    const int P3 = next_pow2(max(nr, 2));
    for (int i = nr + tid; i < P3; i += blockDim.x) keys[i] = 0ull;
    __syncthreads();
    bitonic_sort_desc<false>(keys, P3, tid, blockDim.x);
    const int64_t ob = (q * p.out.parts_total + p.out.part_base) * (int64_t)p.k;
    for (int i = tid; i < p.k; i += blockDim.x) {
        if (i < kk) {
            const uint64_t key = keys[i];
            p.out.scores[ob + i] = key_score(key);
            p.out.labels[ob + i] = p.labels[key_pos(key)];
        } else {
            p.out.scores[ob + i] = 0.f;
            p.out.labels[ob + i] = -1;
        }
    }
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct FlLayout {
    size_t zero_bytes;
    size_t lcnt, lcur, pool_cnt, pool_thr, band, redo_cnt, scanned, loff, nit, ioff, pairq, pairp, items, redo, pool, temp, total;
    size_t temp_bytes;
    int64_t max_items;
};
FlLayout fl_layout(int64_t nq, int P, int k, int nlist) {
    FlLayout L{};
    const int64_t npairs = nq * P;
    size_t o = 0;
    L.lcnt = o; o += align_up(sizeof(int32_t) * ((size_t)nlist + 1), 256);
    L.lcur = o; o += align_up(sizeof(int32_t) * ((size_t)nlist + 1), 256);
    L.pool_cnt = o; o += align_up(sizeof(int32_t) * (size_t)nq * P, 256);
    L.pool_thr = o; o += align_up(sizeof(uint32_t) * (size_t)nq, 256);
    L.band = o; o += align_up(sizeof(float) * (size_t)nq, 256);
    L.redo_cnt = o; o += 256;
    L.scanned = o; o += 256;
    L.zero_bytes = o;
    L.loff = o; o += align_up(sizeof(int32_t) * ((size_t)nlist + 1), 256);
    L.nit = o; o += align_up(sizeof(int32_t) * ((size_t)nlist + 1), 256);
    L.ioff = o; o += align_up(sizeof(int32_t) * ((size_t)nlist + 1), 256);
    L.pairq = o; o += align_up(sizeof(int32_t) * (size_t)npairs, 256);
    L.pairp = o; o += align_up(sizeof(int32_t) * (size_t)npairs, 256);
    L.max_items = npairs / FG + std::min<int64_t>(npairs, nlist) + 1;
    L.items = o; o += align_up(sizeof(int2) * (size_t)L.max_items, 256);
    L.redo = o; o += align_up(sizeof(int2) * (size_t)L.max_items * FG, 256);
    L.pool = o; o += align_up(sizeof(unsigned long long) * (size_t)nq * P * k, 256);
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, (const int32_t*)nullptr, (int32_t*)nullptr, nlist + 1);
    L.temp_bytes = tb + 256;
    L.temp = o; o += align_up(L.temp_bytes, 256);
    L.total = o;
    return L;
}

template <int METRIC>
cudaError_t launch_fl(const IvfFlatScanParams& p, int nlist, void* scratch, int num_sms, cudaStream_t st) {
    const int P = p.nprobe;
    const int64_t npairs = p.nq * P;
    const FlLayout L = fl_layout(p.nq, P, p.k, nlist);
    unsigned char* base = reinterpret_cast<unsigned char*>(scratch);
    int32_t* lcnt = reinterpret_cast<int32_t*>(base + L.lcnt);
    int32_t* lcur = reinterpret_cast<int32_t*>(base + L.lcur);
    int32_t* pool_cnt = reinterpret_cast<int32_t*>(base + L.pool_cnt);
    uint32_t* pool_thr = reinterpret_cast<uint32_t*>(base + L.pool_thr);
    float* band = reinterpret_cast<float*>(base + L.band);
    int32_t* redo_cnt = reinterpret_cast<int32_t*>(base + L.redo_cnt);
    unsigned long long* scanned = reinterpret_cast<unsigned long long*>(base + L.scanned);
    int32_t* loff = reinterpret_cast<int32_t*>(base + L.loff);
    int32_t* nit = reinterpret_cast<int32_t*>(base + L.nit);
    int32_t* ioff = reinterpret_cast<int32_t*>(base + L.ioff);
    int32_t* pairq = reinterpret_cast<int32_t*>(base + L.pairq);
    int32_t* pairp = reinterpret_cast<int32_t*>(base + L.pairp);
    int2* items = reinterpret_cast<int2*>(base + L.items);
    int2* redo = reinterpret_cast<int2*>(base + L.redo);
    unsigned long long* pool = reinterpret_cast<unsigned long long*>(base + L.pool);
    void* temp = base + L.temp;
    size_t tb = L.temp_bytes;

    cudaError_t e = cudaMemsetAsync(base, 0, L.zero_bytes, st);
    if (e != cudaSuccess) return e;
    const unsigned gb = (unsigned)((npairs + 255) / 256), lb = (unsigned)((nlist + 1 + 255) / 256);
    fl_count_kernel<<<gb, 256, 0, st>>>(p.probes, npairs, p.list_off, lcnt, scanned);
    fl_items_per_list_kernel<<<lb, 256, 0, st>>>(lcnt, nlist, nit);
    e = cub::DeviceScan::ExclusiveSum(temp, tb, lcnt, loff, nlist + 1, st);
    if (e != cudaSuccess) return e;
    e = cub::DeviceScan::ExclusiveSum(temp, tb, nit, ioff, nlist + 1, st);
    if (e != cudaSuccess) return e;
    fl_fill_pairs_kernel<<<gb, 256, 0, st>>>(p.probes, npairs, P, p.list_off, loff, lcur, pairq, pairp);
    fl_fill_items_kernel<<<lb, 256, 0, st>>>(nit, ioff, nlist, items);

    FlSeed sd{};
    sd.Q = p.Q; sd.nq = p.nq; sd.dim = p.dim; sd.probes = p.probes; sd.P = P; sd.vecs = p.vecs; sd.dead = p.dead;
    sd.list_off = p.list_off; sd.pool_thr = pool_thr; sd.k = p.k; sd.norms = p.norms; sd.band = band;
    const bool wide = p.dim > 128;
    // k > the sample: no starting threshold, but the sample still measures the slack the hand-over and the final need
    if (wide) ivf_lm_seed_wide_kernel<METRIC><<<(unsigned)((p.nq + 7) / 8), 256, 0, st>>>(sd);
    else ivf_lm_seed_kernel<METRIC><<<(unsigned)((p.nq + 7) / 8), 256, 0, st>>>(sd);

    FlParams sp{};
    sp.Q = p.Q; sp.dim = p.dim; sp.vecs = p.vecs; sp.dead = p.dead; sp.list_off = p.list_off;
    sp.items = items; sp.n_items = ioff + nlist; sp.pair_off = loff; sp.pairq = pairq; sp.pairp = pairp;
    sp.pool = pool; sp.pool_cnt = pool_cnt; sp.pool_thr = pool_thr; sp.pslots = P; sp.k = p.k;
    sp.redo = redo; sp.redo_cnt = redo_cnt; sp.norms = p.norms; sp.band = band;
    if (p.ev_k0) cudaEventRecord(p.ev_k0, st);
    if (wide) {
        const int nchunk = (p.dim + 127) / 128;
        const size_t wsm = (size_t)nchunk * 1024 * sizeof(float2) + (size_t)(FT / 32) * FWR * 16 * sizeof(float);
        e = cudaFuncSetAttribute(ivf_lm_scan_wide_kernel<METRIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsm);
        if (e != cudaSuccess) return e;
        ivf_lm_scan_wide_kernel<METRIC><<<(unsigned)std::min<int64_t>(2 * num_sms, L.max_items), FT, wsm, st>>>(sp, nchunk);
    } else {
        ivf_lm_scan_kernel<METRIC><<<(unsigned)std::min<int64_t>(2 * num_sms, L.max_items), FT, 0, st>>>(sp);
    }
    if (p.ev_k1) cudaEventRecord(p.ev_k1, st);

    FlRedo rd{};
    rd.Q = p.Q; rd.dim = p.dim; rd.vecs = p.vecs; rd.dead = p.dead; rd.list_off = p.list_off; rd.items = items;
    rd.pair_off = loff; rd.pairp = pairp; rd.redo = redo; rd.redo_cnt = redo_cnt; rd.pool = pool; rd.pool_cnt = pool_cnt;
    rd.pslots = P; rd.k = p.k; rd.pool_thr = pool_thr; rd.norms = p.norms;
    ivf_lm_redo_kernel<METRIC><<<(unsigned)(2 * num_sms), 256, sizeof(uint64_t) * FREDO_QCAP + sizeof(float) * p.dim, st>>>(rd);

    FlFinal fp{};
    fp.Q = p.Q; fp.dim = p.dim; fp.vecs = p.vecs; fp.labels = p.labels; fp.pool = pool; fp.pool_cnt = pool_cnt;
    fp.pslots = P; fp.k = p.k; fp.metric = METRIC; fp.out = p.out; fp.norms = p.norms; fp.qnorm = p.qnorm; fp.band = band;
    const size_t fsm = sizeof(uint64_t) * (size_t)next_pow2(std::max(2, P * p.k)) + sizeof(float) * (size_t)p.dim;
    e = cudaFuncSetAttribute(ivf_lm_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsm);
    if (e != cudaSuccess) return e;
    ivf_lm_final_kernel<<<(unsigned)p.nq, 256, fsm, st>>>(fp);
    return cudaGetLastError();
}

}  // namespace

bool ivfflat_lm_supported(int dim, int metric, int nprobe, int k, int64_t nq, int64_t list_total, bool has_budget) {
    if (has_budget || (metric != kL2 && metric != kIP && metric != kCosine)) return false;
    if (dim % 4 != 0 || dim > FW_MAX_DIM || dim < 4) return false;  // d > 128: the wide kernels (queries staged in shared memory)
    if (k < 1 || k > kMaxTopK || (int64_t)nprobe * k > 16384) return false;
    if (nq * nprobe >= ((int64_t)1 << 29) || list_total >= ((int64_t)1 << 32)) return false;
    return true;
}
size_t ivfflat_lm_scratch_bytes(int64_t nq, int nprobe, int k, int nlist) { return fl_layout(nq, nprobe, k, nlist).total; }
int ivfflat_lm_launches() { return 10; }  // count, items-per-list, 2 scans, pair fill, item fill, seed, scan, redo, final

cudaError_t launch_ivfflat_scan_lm(const IvfFlatScanParams& p, int nlist, void* scratch, int num_sms, cudaStream_t st) {
    if (p.nq <= 0) return cudaSuccess;
    if (p.metric == kL2) return launch_fl<kL2>(p, nlist, scratch, num_sms, st);
    if (p.metric == kIP) return launch_fl<kIP>(p, nlist, scratch, num_sms, st);
    return launch_fl<kCosine>(p, nlist, scratch, num_sms, st);
}

cudaError_t ivfflat_lm_scanned_rows(const void* scratch, int64_t nq, int nprobe, int k, int nlist, unsigned long long* out,
                                    cudaStream_t st) {
    const FlLayout L = fl_layout(nq, nprobe, k, nlist);
    cudaError_t e = cudaMemcpyAsync(out, reinterpret_cast<const unsigned char*>(scratch) + L.scanned, sizeof(*out),
                                    cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(st);
}

}  // namespace pyrope
