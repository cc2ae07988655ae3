// build.cu — bit-exact build-time kernels: coarse assignment, PQ encoding, k-means update.
//
// "Centroid assignment and PQ code IDs must be bit-exact given the same trained codebooks": these
// kernels reproduce the reference's fp32 evaluation order (8-lane Vector<float> accumulators,
// separate multiply and add, pairwise horizontal sum — the conventions documented in DESIGN.md) with
// __fmul_rn/__fadd_rn/__fsub_rn so nvcc can never contract them into FMAs.
//   assign : KMeansUtils.FindNearestCentroid  (KMeansUtils.cs:70-93)  via VectorMath.L2Squared /
//            DotProduct / Cosine (VectorMath.cs:8-109)
//   encode : ProductQuantizer.Encode/FindNearest (ProductQuantizer.cs:60-80,122-136) via
//            VectorMath.L2SquaredUnsafe (VectorMath.cs:188-253)
//   update : KMeansUtils.Train mean update (KMeansUtils.cs:46-63)
#include "common.cuh"
#include "exact_arith.cuh"
#include "kernels.h"

#include <float.h>

namespace pyrope {
namespace {

using namespace exact;

// One warp per (vector, subspace): lanes stride over candidates in increasing index order, keep
// the first best (strict '>'), then a warp arg-max that prefers the lower index on ties —
// exactly "lowest index wins" of the sequential reference loops.
// MODE 0: score = -L2Squared (a2)   1: DotProduct (a2)   2: Cosine (a2)   3: -L2SquaredUnsafe (a1)
template <int MODE, typename OutT>
__global__ void __launch_bounds__(256) nearest_exact_kernel(const float* __restrict__ X, int64_t n,
                                                            int64_t ldx, int dd, int nsub,
                                                            const float* __restrict__ Cn, int ncmax,
                                                            const int32_t* __restrict__ ncs,
                                                            const float* __restrict__ cnorms,
                                                            OutT* out) {
    extern __shared__ float vs[];  // [8 warps][dd]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row = (int64_t)blockIdx.x * 8 + warp;
    const int mi = blockIdx.y;
    if (row >= n) return;
    float* v = vs + warp * dd;
    const float* x = X + row * ldx + (int64_t)mi * dd;
    for (int i = lane; i < dd; i += 32) v[i] = x[i];
    __syncwarp();
    const int nc = ncs ? ncs[mi] : ncmax;
    const float* C = Cn + (int64_t)mi * ncmax * dd;
    float vnorm = 0.f;
    if (MODE == 2) vnorm = norm_eval(v, dd);
    float best = -FLT_MAX;
    int besti = 0;
    for (int c = lane; c < nc; c += 32) {
        const float* cv = C + (int64_t)c * dd;
        float s;
        if (MODE == 0) s = -a2_eval<0>(v, cv, dd);
        else if (MODE == 1) s = a2_eval<1>(v, cv, dd);
        else if (MODE == 2) {
            float cn = cnorms[c];
            if (vnorm < 1e-6f || cn < 1e-6f) s = 0.f;
            else s = __fdiv_rn(a2_eval<1>(v, cv, dd), __fmul_rn(vnorm, cn));
        } else s = -a1_l2_eval(v, cv, dd);
        if (s > best) { best = s; besti = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float os = __shfl_xor_sync(0xffffffffu, best, o);
        int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        if (os > best || (os == best && oi < besti)) { best = os; besti = oi; }
    }
    if (lane == 0) out[row * nsub + mi] = (OutT)besti;
}

// Shortlist variant of nearest_exact_kernel: lanes take the (<= 32) shortlisted centroids of the row.
//
// The shortlist holds the k' best 3xTF32 proxy scores p_c (flat_tc.cu: scale_c D + bias_c), so every centroid left out
// has p_j <= plast.  It settles the reference's arg-best when no centroid left out can reach the best re-evaluated one:
// with T_c the exact score in proxy units (L2: 2 x.c - |c|^2 = |x|^2 - |x - c|^2, IP: x.c, Cosine: x.c / |c|), the
// proxy within E_p of T_c and the reference's fp32 score (shifted by |x|^2 for L2, scaled by |x| for Cosine) within E_r,
//     ref_j <= plast + E_p + E_r   and   ref_best >= p0 - E_p - E_r,
// so plast < p0 - 2 (E_p + E_r) puts every left-out centroid strictly below the best (a tie could fall to a lower index
// outside the shortlist: the comparison stays strict).  Both errors are bounded per row from |x| and
// A = max_c |scale_c| |c| (TcOperand.amax; Cauchy-Schwarz: sum|x_i c_i| scale_c <= |x| A):
//   E_p = g_p sum|terms|, g_p = (d + 64) 2^-24: the dropped lo.lo product and the tf32-truncated lo operands (< 1.3 2^-20)
//         plus fp32 accumulation over 3 d / 8 MMA steps (2^-23 each); the slack covers the epilogue's rounding and L2's
//         fp32 |c|^2 bias (sum|terms| <= |x| A + A^2 / 4);
//   E_r = g_r sum|terms|, g_r = fl_gamma(d) (ivf_lm.cu); L2's reference sums (x_i - c_i)^2 <= (|x| + A / 2)^2, Cosine's
//         adds the rounding of the norms and the division (2 g_r |x| A).
// Neither depends on the score: near 0 (centroids orthogonal to the row) a margin relative to the best proxy accepts a
// shortlist whose order is rounding noise.  A Cosine row with |x| < 1e-6 scores 0 against every centroid: index 0.
template <int MODE>
__global__ void __launch_bounds__(256) assign_shortlist_kernel(const float* __restrict__ X, int64_t n, int64_t ldx,
                                                               int dd, const float* __restrict__ C,
                                                               const float* __restrict__ cnorms,
                                                               const float* __restrict__ amax,
                                                               const uint64_t* __restrict__ queue,
                                                               const int32_t* __restrict__ counts, int cap, int kprime,
                                                               int32_t* assign, uint8_t* flag) {
    extern __shared__ float vs[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row = (int64_t)blockIdx.x * 8 + warp;
    if (row >= n) return;
    float* v = vs + warp * dd;
    const float* x = X + row * ldx;
    for (int i = lane; i < dd; i += 32) v[i] = x[i];
    __syncwarp();
    const int c = min(counts[row], 32);
    float vnorm = 0.f;
    if (MODE == 2) vnorm = norm_eval(v, dd);
    float xx = 0.f;
    for (int i = lane; i < dd; i += 32) xx = fmaf(v[i], v[i], xx);
    xx = warp_sum(xx);
    float best = -FLT_MAX;
    int besti = 0x7fffffff;
    float proxy = 0.f;
    if (lane < c) {
        const uint64_t key = __ldcg(queue + row * cap + lane);
        const int cand = (int)key_pos(key);
        proxy = key_score(key);
        const float* cv = C + (int64_t)cand * dd;
        float s;
        if (MODE == 0) s = -a2_eval<0>(v, cv, dd);
        else if (MODE == 1) s = a2_eval<1>(v, cv, dd);
        else {
            float cn = cnorms[cand];
            if (vnorm < 1e-6f || cn < 1e-6f) s = 0.f;
            else s = __fdiv_rn(a2_eval<1>(v, cv, dd), __fmul_rn(vnorm, cn));
        }
        if (s > best) { best = s; besti = cand; }
    }
    // best and worst proxy score of the (unordered) shortlist
    float p0 = lane < c ? proxy : -FLT_MAX, plast = lane < c ? proxy : FLT_MAX;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        p0 = fmaxf(p0, __shfl_xor_sync(0xffffffffu, p0, o));
        plast = fminf(plast, __shfl_xor_sync(0xffffffffu, plast, o));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float os = __shfl_xor_sync(0xffffffffu, best, o);
        int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        if (os > best || (os == best && oi < besti)) { best = os; besti = oi; }
    }
    if (lane == 0) {
        const float A = __ldg(amax), xn = sqrtf(xx) * (1.f + 0x1p-10f);
        const float gp = (float)(dd + 64) * 0x1p-24f, gr = (float)(dd / 4 + 24) * 0x1p-24f;
        float e;
        if (MODE == 0) e = gp * (xn * A + A * A) + gr * (xn + 0.5f * A) * (xn + 0.5f * A);
        else if (MODE == 1) e = (gp + gr) * xn * A;
        else e = (gp + 2.f * gr) * xn * A;
        const float band = 2.f * e * (1.f + 0x1p-10f);
        const bool zero_row = MODE == 2 && vnorm < 1e-6f;
        const bool incomplete = !zero_row && ((c == 0) || besti == 0x7fffffff || (c >= kprime && !(plast < p0 - band)));
        assign[row] = incomplete || zero_row ? 0 : besti;
        flag[row] = incomplete ? 1 : 0;
    }
}

__global__ void scatter_i32_kernel(const int32_t* src, const int64_t* idx, int64_t n, int32_t* dst) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[idx[i]] = src[i];
}

// Coarse ranking in the reference's arithmetic: the fast coarse stage hands P_in >= P_out candidate lists per
// query; their scores are recomputed exactly as IvfFlatVectorIndex.cs:186-193 / IvfPqVectorIndex.cs:141-147 do
// (VectorMath.L2Squared / DotProduct / Cosine, single 8-lane accumulator) and the best P_out are emitted in
// descending order (ties to the lower list index), so the probed set equals the oracle's even when two
// centroids score within a rounding error of each other.  One CTA per query.
//
// The stage-one scores (fp32, another summation order) settle the probed SET when the P_out-th and (P_out+1)-th are
// further apart than both their errors.  For L2 the summed terms are non-negative and the error is relative to the
// score; for IP and Cosine it is gamma * sum|q_i c_i|, at most gamma |q| |c| (Cosine: gamma), whatever the score, so near
// 0 (centroids orthogonal to the query) a relative margin settles nothing.  When even the last candidate lies within
// that band of the P_out-th, a centroid the stage left out may belong to the set: every centroid is ranked exactly.
template <int METRIC>
__global__ void __launch_bounds__(128) coarse_rerank_kernel(const float* __restrict__ Q, int dim,
                                                            const float* __restrict__ C, const float* __restrict__ cnorms,
                                                            int nc, const int64_t* __restrict__ pin,
                                                            const float* __restrict__ sin, int P_in,
                                                            int64_t* pout, float* sout, int P_out, int Psort, int H,
                                                            int need_order) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem_raw);   // [max(Psort, 2 H)]
    float* qs = reinterpret_cast<float*>(keys + max(Psort, 2 * H));  // [dim]
    __shared__ float s_qn;
    __shared__ unsigned s_cmax;
    const int64_t q = blockIdx.x;
    const int tid = threadIdx.x;
    // L2 fast path: the stage-one scores (accurate to ~1e-6 relative, sorted descending) already separate the
    // P_out-th from the (P_out+1)-th candidate by far more than their rounding error, so the probed SET is settled;
    // unless the caller needs the exact order too (MaxScans budgets walk lists in rank order), copy.
    if (METRIC == 0 && !need_order && sin && !sout) {
        bool settled = P_in <= P_out;
        if (!settled) {
            const float a = sin[q * P_in + P_out - 1], b = sin[q * P_in + P_out];
            settled = pin[q * P_in + P_out] < 0 || (a - b) > 2e-5f * fmaxf(fabsf(a), fabsf(b)) + 1e-30f;
        }
        if (settled) {  // block-uniform
            for (int i = tid; i < P_out; i += blockDim.x) pout[q * P_out + i] = i < P_in ? pin[q * P_in + i] : -1;
            return;
        }
    }
    for (int d = tid; d < dim; d += blockDim.x) qs[d] = Q[q * dim + d];
    if (tid == 0) s_cmax = 0u;
    __syncthreads();
    if (METRIC != 0 && tid == 0) s_qn = norm_eval(qs, dim);
    bool exhaustive = false;
    if (METRIC != 0 && sin && P_in > P_out) {
        if (METRIC == 1) {  // |c| of the candidates (fp32, rounded up below)
            for (int i = tid; i < P_in; i += blockDim.x) {
                const int64_t l = pin[q * P_in + i];
                if (l >= 0) atomicMax(&s_cmax, __float_as_uint(norm_eval(C + l * dim, dim)));
            }
        }
        __syncthreads();
        // two orders of at most dim terms differ by <= (dim / 4 + 24) 2^-24 sum|term| (as ivf_lm.cu's fl_gamma)
        const float gam = (float)(dim / 4 + 24) * 0x1p-24f;
        const float e = METRIC == 2 ? gam : gam * s_qn * __uint_as_float(s_cmax) * (1.f + 0x1p-10f);
        const float a = sin[q * P_in + P_out - 1], b = sin[q * P_in + P_out], last = sin[q * P_in + P_in - 1];
        exhaustive = P_in < nc && pin[q * P_in + P_in - 1] >= 0 && last >= a - 2.f * e - 1e-30f;
        if (!exhaustive && !need_order && !sout && (pin[q * P_in + P_out] < 0 || a - b > 2.f * e + 1e-30f)) {
            for (int i = tid; i < P_out; i += blockDim.x) pout[q * P_out + i] = pin[q * P_in + i];
            return;  // block-uniform
        }
    }
    __syncthreads();
    auto exact_key = [&](int64_t l) -> uint64_t {
        const float* cv = C + l * dim;
        float s;
        if (METRIC == 0) s = -a2_eval<0>(qs, cv, dim);
        else if (METRIC == 1) s = a2_eval<1>(qs, cv, dim);
        else {
            const float cn = cnorms[l];
            s = (s_qn < 1e-6f || cn < 1e-6f) ? 0.f : __fdiv_rn(a2_eval<1>(qs, cv, dim), __fmul_rn(s_qn, cn));
        }
        return make_key(s, (uint32_t)l);
    };
    int P;
    if (exhaustive) {  // every centroid, H at a time, merged into the best H
        P = 2 * H;
        for (int i = tid; i < H; i += blockDim.x) keys[i] = 0ull;
        for (int c0 = 0; c0 < nc; c0 += H) {
            for (int i = tid; i < H; i += blockDim.x) keys[H + i] = c0 + i < nc ? exact_key(c0 + i) : 0ull;
            __syncthreads();
            bitonic_sort_desc<false>(keys, P, tid, blockDim.x);
            __syncthreads();
        }
    } else {
        P = Psort;
        for (int i = tid; i < Psort; i += blockDim.x) {
            const int64_t l = i < P_in ? pin[q * P_in + i] : -1;
            keys[i] = l >= 0 ? exact_key(l) : 0ull;
        }
        __syncthreads();
        bitonic_sort_desc<false>(keys, P, tid, blockDim.x);
        __syncthreads();
    }
    for (int i = tid; i < P_out; i += blockDim.x) {
        const uint64_t key = i < P ? keys[i] : 0ull;
        pout[q * P_out + i] = key ? (int64_t)key_pos(key) : -1;
        if (sout) sout[q * P_out + i] = key ? key_score(key) : 0.f;
    }
}

__global__ void row_norms_kernel(const float* X, int64_t n, int dim, int64_t ldx, float* out) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    out[r] = norm_eval(X + r * ldx, dim);
}

__global__ void residual_kernel(const float* X, int64_t n, int dim, const float* C, const int32_t* assign,
                                float* out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * dim) return;
    int64_t r = i / dim;
    int d = (int)(i - r * dim);
    out[i] = __fsub_rn(X[i], C[(int64_t)assign[r] * dim + d]);
}

// one CTA per cluster; thread per dimension keeps the running fp32 sum in data order
__global__ void __launch_bounds__(128) kmeans_update_kernel(const float* __restrict__ X, int64_t ldx, int dim,
                                                            const int64_t* __restrict__ offs,
                                                            const int32_t* __restrict__ order,
                                                            float* centroids, int* changed) {
    const int c = blockIdx.x;
    const int64_t b = offs[c], e = offs[c + 1];
    if (e == b) return;  // empty cluster keeps its centroid (KMeansUtils.cs:48)
    const float fc = (float)(int)(e - b);
    int differs = 0;
    // pass 1: decide whether any dimension moved by more than 1e-6 (ArraysEqual :95-101)
    for (int d0 = 0; d0 < dim; d0 += blockDim.x) {
        int d = d0 + threadIdx.x;
        if (d < dim) {
            float s = 0.f;
            for (int64_t j = b; j < e; ++j) s = __fadd_rn(s, __ldg(X + (int64_t)order[j] * ldx + d));
            float nv = __fdiv_rn(s, fc);
            float df = __fsub_rn(centroids[(int64_t)c * dim + d], nv);
            if ((double)fabsf(df) > 1e-6) differs = 1;
        }
    }
    differs = __syncthreads_or(differs);
    if (!differs) return;
    for (int d0 = 0; d0 < dim; d0 += blockDim.x) {
        int d = d0 + threadIdx.x;
        if (d < dim) {
            float s = 0.f;
            for (int64_t j = b; j < e; ++j) s = __fadd_rn(s, __ldg(X + (int64_t)order[j] * ldx + d));
            centroids[(int64_t)c * dim + d] = __fdiv_rn(s, fc);
        }
    }
    if (threadIdx.x == 0) *changed = 1;
}

__global__ void gather_rows_kernel(const uint8_t* X, int64_t row_bytes, const int64_t* idx, int64_t n,
                                   uint8_t* out) {
    // one warp per row; 16-byte words when aligned
    int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (r >= n) return;
    const uint8_t* src = X + idx[r] * row_bytes;
    uint8_t* dst = out + r * row_bytes;
    if ((row_bytes & 15) == 0 && ((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0) {
        const uint4* s4 = reinterpret_cast<const uint4*>(src);
        uint4* d4 = reinterpret_cast<uint4*>(dst);
        for (int64_t i = lane; i < row_bytes / 16; i += 32) d4[i] = s4[i];
    } else {
        for (int64_t i = lane; i < row_bytes; i += 32) dst[i] = src[i];
    }
}

// scatter rows: out[idx[r]] = X[r]
__global__ void scatter_rows_kernel(const uint8_t* X, int64_t row_bytes, const int64_t* idx, int64_t n,
                                    uint8_t* out) {
    int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (r >= n) return;
    const uint8_t* src = X + r * row_bytes;
    uint8_t* dst = out + idx[r] * row_bytes;
    if ((row_bytes & 15) == 0 && ((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0) {
        const uint4* s4 = reinterpret_cast<const uint4*>(src);
        uint4* d4 = reinterpret_cast<uint4*>(dst);
        for (int64_t i = lane; i < row_bytes / 16; i += 32) d4[i] = s4[i];
    } else {
        for (int64_t i = lane; i < row_bytes; i += 32) dst[i] = src[i];
    }
}

// where[i] = position in the ascending array `sorted` (ns entries) holding labels[i], or -1; entries whose
// skip byte is non-zero are not looked up.  Compaction uses it to find the tail rows a moved head id replaces.
__global__ void find_labels_kernel(const int64_t* __restrict__ labels, const uint8_t* __restrict__ skip, int64_t n,
                                   const int64_t* __restrict__ sorted, int64_t ns, int64_t* __restrict__ where) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t hit = -1;
    if (!skip || !skip[i]) {
        const int64_t v = labels[i];
        int64_t lo = 0, hi = ns;
        while (lo < hi) {
            int64_t mid = (lo + hi) >> 1;
            if (sorted[mid] < v) lo = mid + 1; else hi = mid;
        }
        if (lo < ns && sorted[lo] == v) hit = lo;
    }
    where[i] = hit;
}

__global__ void iota64_kernel(int64_t* out, int64_t n, int64_t base) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = base + i;
}

// counter-based uniform [0,1) generator (splitmix64 finaliser), 24 random mantissa bits
__global__ void fill_uniform_kernel(float* out, int64_t n, uint64_t seed, uint64_t offset) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t z = (offset + (uint64_t)i) * 0x9E3779B97F4A7C15ull + seed;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z = z ^ (z >> 31);
    out[i] = (float)(uint32_t)(z >> 40) * (1.0f / 16777216.0f);
}

inline unsigned blocks_for(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

}  // namespace

cudaError_t launch_assign_exact(int metric, int dim, int64_t n, const float* X, int64_t ldx, int nc,
                                const float* centroids, const float* cnorms, int32_t* assign,
                                cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    dim3 grid(blocks_for(n, 8), 1);
    size_t smem = sizeof(float) * 8 * (size_t)dim;
    cudaError_t e = cudaSuccess;
#define PYROPE_LAUNCH_NEAREST(MODE)                                                                  \
    if (smem > 48 * 1024)                                                                            \
        e = cudaFuncSetAttribute(nearest_exact_kernel<MODE, int32_t>,                                \
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);            \
    if (e != cudaSuccess) return e;                                                                  \
    nearest_exact_kernel<MODE, int32_t><<<grid, 256, smem, st>>>(X, n, ldx, dim, 1, centroids, nc,   \
                                                                  nullptr, cnorms, assign);
    if (metric == kL2) { PYROPE_LAUNCH_NEAREST(0) }
    else if (metric == kIP) { PYROPE_LAUNCH_NEAREST(1) }
    else { PYROPE_LAUNCH_NEAREST(2) }
#undef PYROPE_LAUNCH_NEAREST
    return cudaGetLastError();
}

cudaError_t launch_assign_from_shortlist(int metric, int dim, int64_t n, const float* X, int64_t ldx,
                                         const float* centroids, const float* cnorms, const float* amax,
                                         const uint64_t* queue, const int32_t* counts, int cap, int kprime,
                                         int32_t* assign, uint8_t* flag, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const unsigned grid = blocks_for(n, 8);
    const size_t smem = sizeof(float) * 8 * (size_t)dim;
    if (metric == kL2)
        assign_shortlist_kernel<0><<<grid, 256, smem, st>>>(X, n, ldx, dim, centroids, cnorms, amax, queue, counts, cap, kprime, assign, flag);
    else if (metric == kIP)
        assign_shortlist_kernel<1><<<grid, 256, smem, st>>>(X, n, ldx, dim, centroids, cnorms, amax, queue, counts, cap, kprime, assign, flag);
    else
        assign_shortlist_kernel<2><<<grid, 256, smem, st>>>(X, n, ldx, dim, centroids, cnorms, amax, queue, counts, cap, kprime, assign, flag);
    return cudaGetLastError();
}

cudaError_t launch_scatter_i32(const int32_t* src, const int64_t* idx, int64_t n, int32_t* dst, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    scatter_i32_kernel<<<blocks_for(n, 256), 256, 0, st>>>(src, idx, n, dst);
    return cudaGetLastError();
}

cudaError_t launch_coarse_rerank_exact(int metric, int dim, int64_t nq, const float* Q, const float* centroids,
                                       const float* cnorms, int nc, const int64_t* probes_in, const float* scores_in, int P_in,
                                       int64_t* probes_out, float* scores_out, int P_out, int need_order, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    const int Psort = next_pow2(P_in < 2 ? 2 : P_in);
    const int H = metric == kL2 ? 0 : next_pow2(P_out < 64 ? 64 : P_out);  // the exhaustive ranking's merge width
    const size_t smem = sizeof(uint64_t) * (size_t)std::max(Psort, 2 * H) + sizeof(float) * (size_t)dim;
    if (smem > 48 * 1024) return cudaErrorInvalidValue;
    if (metric == kL2)
        coarse_rerank_kernel<0><<<(unsigned)nq, 128, smem, st>>>(Q, dim, centroids, cnorms, nc, probes_in, scores_in, P_in, probes_out, scores_out, P_out, Psort, H, need_order);
    else if (metric == kIP)
        coarse_rerank_kernel<1><<<(unsigned)nq, 128, smem, st>>>(Q, dim, centroids, cnorms, nc, probes_in, scores_in, P_in, probes_out, scores_out, P_out, Psort, H, need_order);
    else
        coarse_rerank_kernel<2><<<(unsigned)nq, 128, smem, st>>>(Q, dim, centroids, cnorms, nc, probes_in, scores_in, P_in, probes_out, scores_out, P_out, Psort, H, need_order);
    return cudaGetLastError();
}

cudaError_t launch_pq_encode_exact(const float* R, int64_t n, int dim, int m, int kpad,
                                   const float* codebook, const int32_t* ksub, uint8_t* codes,
                                   cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const int sub = dim / m;
    dim3 grid(blocks_for(n, 8), (unsigned)m);
    size_t smem = sizeof(float) * 8 * (size_t)sub;
    nearest_exact_kernel<3, uint8_t><<<grid, 256, smem, st>>>(R, n, dim, sub, m, codebook, kpad, ksub,
                                                              nullptr, codes);
    return cudaGetLastError();
}

cudaError_t launch_row_norms_exact(const float* X, int64_t n, int dim, int64_t ldx, float* out,
                                   cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    row_norms_kernel<<<blocks_for(n, 128), 128, 0, st>>>(X, n, dim, ldx, out);
    return cudaGetLastError();
}

cudaError_t launch_residuals(const float* X, int64_t n, int dim, const float* centroids,
                             const int32_t* assign, float* out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    residual_kernel<<<blocks_for(n * dim, 256), 256, 0, st>>>(X, n, dim, centroids, assign, out);
    return cudaGetLastError();
}

cudaError_t launch_kmeans_update(const float* X, int64_t ldx, int dim, int nc, const int64_t* offs,
                                 const int32_t* order, float* centroids, int* changed, cudaStream_t st) {
    if (nc <= 0) return cudaSuccess;
    kmeans_update_kernel<<<(unsigned)nc, 128, 0, st>>>(X, ldx, dim, offs, order, centroids, changed);
    return cudaGetLastError();
}

cudaError_t launch_gather_rows(const void* X, int64_t row_bytes, const int64_t* idx, int64_t n, void* out,
                               cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    gather_rows_kernel<<<blocks_for(n * 32, 256), 256, 0, st>>>((const uint8_t*)X, row_bytes, idx, n,
                                                               (uint8_t*)out);
    return cudaGetLastError();
}

cudaError_t launch_scatter_rows(const void* X, int64_t row_bytes, const int64_t* idx, int64_t n, void* out,
                                cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    scatter_rows_kernel<<<blocks_for(n * 32, 256), 256, 0, st>>>((const uint8_t*)X, row_bytes, idx, n,
                                                                (uint8_t*)out);
    return cudaGetLastError();
}

cudaError_t launch_find_labels(const int64_t* labels, const uint8_t* skip, int64_t n, const int64_t* sorted,
                               int64_t ns, int64_t* where, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    find_labels_kernel<<<blocks_for(n, 256), 256, 0, st>>>(labels, skip, n, sorted, ns, where);
    return cudaGetLastError();
}

cudaError_t launch_iota64(int64_t* out, int64_t n, int64_t base, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    iota64_kernel<<<blocks_for(n, 256), 256, 0, st>>>(out, n, base);
    return cudaGetLastError();
}

cudaError_t launch_fill_uniform(float* out, int64_t n, uint64_t seed, uint64_t offset, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    fill_uniform_kernel<<<blocks_for(n, 256), 256, 0, st>>>(out, n, seed, offset);
    return cudaGetLastError();
}

}  // namespace pyrope
