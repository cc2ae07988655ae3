// flat.cu — K1 exact FLAT scan with fused top-k (CUDA-core path) and K6 merge.
//
// Replaces BruteForceVectorIndex.Search's scan loop (BruteForceVectorIndex.cs:341-360: one
// L2SquaredUnsafe/DotProductUnsafe + heap push per row per query) with a batched, register-tiled
// score kernel that never materialises the Q x N score matrix: each CTA owns 64 queries and a
// range of 128-row base tiles, filters scores against a per-query running threshold and keeps
// candidates in a per-(split,query) queue that is pruned to the best k whenever it may overflow.
#include "common.cuh"
#include "kernels.h"

namespace pyrope {

namespace {

constexpr int TQ = 64;    // queries per CTA
constexpr int TN = 128;   // base rows per tile
constexpr int TK = 16;    // k-chunk
constexpr int NT = 256;   // threads

__device__ __forceinline__ float4 load4_guard(const float* base, int64_t row, int64_t nrows,
                                              int64_t ld, int col, int dim, bool vec_ok) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < nrows) {
        const float* p = base + row * ld + col;
        if (vec_ok) {
            if (col < dim) v = __ldg(reinterpret_cast<const float4*>(p));
        } else {
            if (col + 0 < dim) v.x = __ldg(p + 0);
            if (col + 1 < dim) v.y = __ldg(p + 1);
            if (col + 2 < dim) v.z = __ldg(p + 2);
            if (col + 3 < dim) v.w = __ldg(p + 3);
        }
    }
    return v;
}

template <int METRIC>
__device__ __forceinline__ void mac(float& acc, float q, float x) {
    if (METRIC == kL2) {
        float d = q - x;
        acc = fmaf(d, d, acc);
    } else {
        acc = fmaf(q, x, acc);
    }
}

template <int METRIC>
__global__ void __launch_bounds__(NT) flat_scan_kernel(FlatScanParams p, int64_t ntiles,
                                                       int64_t tiles_per_split, int nsort) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* Qs = reinterpret_cast<float*>(smem_raw);                 // [TK][TQ]
    float* Xs = Qs + TK * TQ;                                        // [TK][TN]
    uint64_t* thr = reinterpret_cast<uint64_t*>(Xs + TK * TN);       // [TQ]
    int* cnt = reinterpret_cast<int*>(thr + TQ);                     // [TQ]
    int* need = cnt + TQ;                                            // [2]
    uint64_t* stage = reinterpret_cast<uint64_t*>(need + 2);         // [nsort][cap]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid & 15, ty = tid >> 4;
    const int64_t q0 = (int64_t)blockIdx.x * TQ;
    const int split = blockIdx.y;
    const int dim = p.dim;
    const bool vec_ok = (dim % 4 == 0);
    const int cap = p.cap, k = p.k;

    for (int i = tid; i < TQ; i += NT) { thr[i] = 0; cnt[i] = 0; }
    if (tid == 0) need[0] = 0;
    __syncthreads();

    const int64_t t_begin = (int64_t)split * tiles_per_split;
    const int64_t t_end = min(ntiles, t_begin + tiles_per_split);
    uint64_t* myq = p.queue + ((int64_t)split * p.nq) * cap;

    // loader coordinates
    const int qrow = tid & 63, qc4 = tid >> 6;            // Q tile: 64 rows x 4 float4
    const int xrow = tid & 127, xc4 = tid >> 7;           // X tile: 128 rows x 4 float4 (2 per thread)

    auto sort_query = [&](int qi, int w, bool final) {
        const int64_t gq = q0 + qi;
        uint64_t* st = stage + (int64_t)w * cap;
        uint64_t* g = myq + gq * cap;
        int c = min(cnt[qi], cap);
        int P = next_pow2(max(c, 2));
        for (int i = lane; i < P; i += 32) st[i] = i < c ? g[i] : 0ull;
        __syncwarp();
        bitonic_sort_desc<true>(st, P, lane, 32);
        int keep = min(c, k);
        if (!final) {
            for (int i = lane; i < keep; i += 32) g[i] = st[i];
            if (lane == 0) { cnt[qi] = keep; thr[qi] = (keep == k) ? st[k - 1] : 0ull; }
        } else {
            float* os = p.out.scores + (gq * p.out.parts_total + p.out.part_base + split) * (int64_t)k;
            int64_t* ol = p.out.labels + (gq * p.out.parts_total + p.out.part_base + split) * (int64_t)k;
            for (int i = lane; i < k; i += 32) {
                if (i < keep) {
                    uint64_t key = st[i];
                    uint32_t pos = key_pos(key);
                    os[i] = key_score(key);
                    ol[i] = p.labels ? p.labels[pos] : (int64_t)pos;
                } else {
                    os[i] = 0.f;
                    ol[i] = -1;
                }
            }
        }
        __syncwarp();
    };

    for (int64_t t = t_begin; t < t_end; ++t) {
        const int64_t n0 = t * TN;
        float acc[4][8];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

        float4 qreg = load4_guard(p.Q, q0 + qrow, p.nq, dim, qc4 * 4, dim, vec_ok);
        float4 xr0 = load4_guard(p.X, n0 + xrow, p.n_scan, dim, xc4 * 4, dim, vec_ok);
        float4 xr1 = load4_guard(p.X, n0 + xrow, p.n_scan, dim, (xc4 + 2) * 4, dim, vec_ok);

        for (int k0 = 0; k0 < dim; k0 += TK) {
            __syncthreads();  // previous chunk consumed
            {
                int c = qc4 * 4;
                Qs[(c + 0) * TQ + qrow] = qreg.x; Qs[(c + 1) * TQ + qrow] = qreg.y;
                Qs[(c + 2) * TQ + qrow] = qreg.z; Qs[(c + 3) * TQ + qrow] = qreg.w;
                c = xc4 * 4;
                Xs[(c + 0) * TN + xrow] = xr0.x; Xs[(c + 1) * TN + xrow] = xr0.y;
                Xs[(c + 2) * TN + xrow] = xr0.z; Xs[(c + 3) * TN + xrow] = xr0.w;
                c = (xc4 + 2) * 4;
                Xs[(c + 0) * TN + xrow] = xr1.x; Xs[(c + 1) * TN + xrow] = xr1.y;
                Xs[(c + 2) * TN + xrow] = xr1.z; Xs[(c + 3) * TN + xrow] = xr1.w;
            }
            __syncthreads();
            if (k0 + TK < dim) {  // prefetch next chunk while computing this one
                int kn = k0 + TK;
                qreg = load4_guard(p.Q, q0 + qrow, p.nq, dim, kn + qc4 * 4, dim, vec_ok);
                xr0 = load4_guard(p.X, n0 + xrow, p.n_scan, dim, kn + xc4 * 4, dim, vec_ok);
                xr1 = load4_guard(p.X, n0 + xrow, p.n_scan, dim, kn + (xc4 + 2) * 4, dim, vec_ok);
            }
#pragma unroll
            for (int kk = 0; kk < TK; ++kk) {
                float4 q4 = *reinterpret_cast<const float4*>(&Qs[kk * TQ + ty * 4]);
                float4 xa = *reinterpret_cast<const float4*>(&Xs[kk * TN + tx * 4]);
                float4 xb = *reinterpret_cast<const float4*>(&Xs[kk * TN + 64 + tx * 4]);
                float qv[4] = {q4.x, q4.y, q4.z, q4.w};
                float xv[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) mac<METRIC>(acc[i][j], qv[i], xv[j]);
            }
        }

        // ---- epilogue: score, filter against the running threshold, enqueue
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int rl = (j < 4) ? (tx * 4 + j) : (64 + tx * 4 + (j - 4));
            int64_t pos = n0 + rl;
            bool ok = pos < p.n_scan;
            if (ok && p.dead) ok = (p.dead[pos] == 0);
            float xn = 0.f;
            if (METRIC == kCosine && ok) xn = p.xnorm[pos];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                int qi = ty * 4 + i;
                int64_t gq = q0 + qi;
                if (!ok || gq >= p.nq) continue;
                float s;
                if (METRIC == kL2) s = -acc[i][j];
                else if (METRIC == kIP) s = acc[i][j];
                else {
                    float qn = p.qnorm[gq];
                    s = (qn < 1e-6f || xn < 1e-6f) ? 0.f : acc[i][j] / (qn * xn);
                }
                uint64_t key = make_key(s, (uint32_t)pos);
                if (key > thr[qi]) {
                    int slot = atomicAdd(&cnt[qi], 1);
                    if (slot < cap) myq[gq * cap + slot] = key;
                    if (slot + 1 > cap - TN) need[0] = 1;
                }
            }
        }
        __syncthreads();
        if (need[0]) {
            if (warp < nsort) {
                for (int qi = warp; qi < TQ; qi += nsort)
                    if (q0 + qi < p.nq && cnt[qi] > cap - TN) sort_query(qi, warp, false);
            }
            __syncthreads();
            if (tid == 0) need[0] = 0;
        }
    }

    __syncthreads();
    if (warp < nsort) {
        for (int qi = warp; qi < TQ; qi += nsort)
            if (q0 + qi < p.nq) sort_query(qi, warp, true);
    }
}

// ------------------------------------------------------------------------------------------
// K6 merge: one CTA per query; parts*k_in candidates -> k_out.
// PER_Q: query q keeps only entries j < k_q = k_per_query[q] of every part (the rest count as empty, for the
// de-duplication too) and its output is cut at k_q — what the same merge with k_in = k_out = k_q gives, because the
// sort key (score, part * k_in + j) orders candidates alike for any k_in.
// ------------------------------------------------------------------------------------------
template <bool PER_Q>
__global__ void __launch_bounds__(256) merge_pairs_kernel(int64_t nq, int parts, int k_in, int k_out,
                                                          const float* __restrict__ in_s,
                                                          const int64_t* __restrict__ in_l,
                                                          int64_t part_stride, int64_t q_stride,
                                                          float* out_s, int64_t* out_l,
                                                          int32_t* out_c, int P, int dedupe,
                                                          const int32_t* __restrict__ k_per_query) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem_raw);
    __shared__ int s_count;
    const int64_t q = blockIdx.x;
    const int tid = threadIdx.x;
    const int total = parts * k_in;
    const int kq = PER_Q ? min(k_per_query[q], k_in) : k_in;
    const int kcut = PER_Q ? min(kq, k_out) : k_out;
    if (tid == 0) s_count = 0;
    for (int i = tid; i < P; i += blockDim.x) {
        uint64_t key = 0;
        if (i < total) {
            int part = i / k_in, j = i - part * k_in;
            int64_t a = part * part_stride + q * q_stride + j;
            const int64_t lab = (!PER_Q || j < kq) ? in_l[a] : -1;
            if (lab >= 0) {
                bool dup = false;
                if (dedupe) {  // the same id in a lower part (the head) wins
                    for (int pp = 0; pp < part && !dup; ++pp) {
                        const int64_t b = pp * part_stride + q * q_stride;
                        for (int jj = 0; jj < kq; ++jj)
                            if (in_l[b + jj] == lab) { dup = true; break; }
                    }
                }
                if (!dup) key = make_key(in_s[a], (uint32_t)i);
            }
        }
        keys[i] = key;
    }
    __syncthreads();
    bitonic_sort_desc<false>(keys, P, tid, blockDim.x);
    int local = 0;
    for (int i = tid; i < k_out; i += blockDim.x) {
        uint64_t key = (i < P && (!PER_Q || i < kcut)) ? keys[i] : 0ull;
        if (key) {
            int idx = (int)key_pos(key);
            int part = idx / k_in, j = idx - part * k_in;
            int64_t a = part * part_stride + q * q_stride + j;
            out_s[q * k_out + i] = in_s[a];
            out_l[q * k_out + i] = in_l[a];
            ++local;
        } else {
            out_s[q * k_out + i] = 0.f;
            out_l[q * k_out + i] = -1;
        }
    }
    if (local) atomicAdd(&s_count, local);
    __syncthreads();
    if (tid == 0 && out_c) out_c[q] = s_count;
}

// Few candidates per query (the multi-GPU merge: ranks x k): one WARP per query, eight queries per CTA, no block barriers.
// PER_Q as for merge_pairs_kernel.
template <bool PER_Q>
__global__ void __launch_bounds__(256) merge_pairs_warp_kernel(int64_t nq, int parts, int k_in, int k_out,
                                                               const float* __restrict__ in_s,
                                                               const int64_t* __restrict__ in_l,
                                                               int64_t part_stride, int64_t q_stride,
                                                               float* out_s, int64_t* out_l,
                                                               int32_t* out_c, int P, int dedupe,
                                                               const int32_t* __restrict__ k_per_query) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem_raw) + (size_t)warp * P;
    const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (q >= nq) return;
    const int total = parts * k_in;
    const int kq = PER_Q ? min(k_per_query[q], k_in) : k_in;
    const int kcut = PER_Q ? min(kq, k_out) : k_out;
    for (int i = lane; i < P; i += 32) {
        uint64_t key = 0;
        if (i < total) {
            const int part = i / k_in, j = i - part * k_in;
            const int64_t a = part * part_stride + q * q_stride + j;
            const int64_t lab = (!PER_Q || j < kq) ? in_l[a] : -1;
            if (lab >= 0) {
                bool dup = false;
                if (dedupe) {  // the same id in a lower part (the head) wins
                    for (int pp = 0; pp < part && !dup; ++pp) {
                        const int64_t b = pp * part_stride + q * q_stride;
                        for (int jj = 0; jj < kq; ++jj)
                            if (in_l[b + jj] == lab) { dup = true; break; }
                    }
                }
                if (!dup) key = make_key(in_s[a], (uint32_t)i);
            }
        }
        keys[i] = key;
    }
    __syncwarp();
    bitonic_sort_desc<true>(keys, P, lane, 32);
    int local = 0;
    for (int i = lane; i < k_out; i += 32) {
        const uint64_t key = (i < P && (!PER_Q || i < kcut)) ? keys[i] : 0ull;
        if (key) {
            const int idx = (int)key_pos(key);
            const int part = idx / k_in, j = idx - part * k_in;
            const int64_t a = part * part_stride + q * q_stride + j;
            out_s[q * k_out + i] = in_s[a];
            out_l[q * k_out + i] = in_l[a];
            ++local;
        } else {
            out_s[q * k_out + i] = 0.f;
            out_l[q * k_out + i] = -1;
        }
    }
    local = __reduce_add_sync(0xffffffffu, local);
    if (lane == 0 && out_c) out_c[q] = local;
}

}  // namespace

int flat_scan_cap(int k) {
    int c = next_pow2(k + TN);
    return c < 256 ? 256 : c;
}

int flat_scan_pick_splits(int64_t nq, int64_t n_scan, int k, int num_sms, int max_parts) {
    int64_t qtiles = (nq + TQ - 1) / TQ;
    int64_t ntiles = (n_scan + TN - 1) / TN;
    if (ntiles < 1) ntiles = 1;
    int64_t want = (2 * (int64_t)num_sms + qtiles - 1) / qtiles;  // ~2 CTAs per SM overall
    int64_t lim = kMergeMaxCandidates / (k > 0 ? k : 1);
    if (max_parts > 0 && lim > max_parts) lim = max_parts;
    if (want > lim) want = lim;
    if (want > ntiles) want = ntiles;
    if (want < 1) want = 1;
    return (int)want;
}

cudaError_t launch_flat_scan(const FlatScanParams& p, cudaStream_t st) {
    if (p.nq <= 0) return cudaSuccess;
    int64_t ntiles = (p.n_scan + TN - 1) / TN;
    int64_t tps = (ntiles + p.splits - 1) / p.splits;
    if (tps < 1) tps = 1;
    int nsort = 4096 / p.cap;
    if (nsort > NT / 32) nsort = NT / 32;
    if (nsort < 1) nsort = 1;
    size_t smem = sizeof(float) * (TK * TQ + TK * TN) + sizeof(uint64_t) * TQ + sizeof(int) * (TQ + 2) +
                  sizeof(uint64_t) * (size_t)nsort * p.cap;
    dim3 grid((unsigned)((p.nq + TQ - 1) / TQ), (unsigned)p.splits);
    switch (p.metric) {
        case kL2: flat_scan_kernel<kL2><<<grid, NT, smem, st>>>(p, ntiles, tps, nsort); break;
        case kIP: flat_scan_kernel<kIP><<<grid, NT, smem, st>>>(p, ntiles, tps, nsort); break;
        default: flat_scan_kernel<kCosine><<<grid, NT, smem, st>>>(p, ntiles, tps, nsort); break;
    }
    return cudaGetLastError();
}

cudaError_t launch_merge_pairs(int64_t nq, int parts, int k_in, int k_out, const float* in_scores,
                               const int64_t* in_labels, int64_t part_stride, int64_t q_stride,
                               float* out_scores, int64_t* out_labels, int32_t* out_counts,
                               cudaStream_t st, bool dedupe, const int32_t* k_per_query) {
    if (nq <= 0) return cudaSuccess;
    int total = parts * k_in;
    if (total > kMergeMaxCandidates) return cudaErrorInvalidValue;
    int P = next_pow2(total < 2 ? 2 : total);
    if (P <= 256) {
        const unsigned grid = (unsigned)((nq + 7) / 8);
        const size_t smem = sizeof(uint64_t) * (size_t)P * 8;
        if (k_per_query)
            merge_pairs_warp_kernel<true><<<grid, 256, smem, st>>>(nq, parts, k_in, k_out, in_scores, in_labels, part_stride,
                                                                  q_stride, out_scores, out_labels, out_counts, P,
                                                                  dedupe ? 1 : 0, k_per_query);
        else
            merge_pairs_warp_kernel<false><<<grid, 256, smem, st>>>(nq, parts, k_in, k_out, in_scores, in_labels, part_stride,
                                                                   q_stride, out_scores, out_labels, out_counts, P,
                                                                   dedupe ? 1 : 0, nullptr);
        return cudaGetLastError();
    }
    const size_t smem = sizeof(uint64_t) * (size_t)P;
    if (k_per_query)
        merge_pairs_kernel<true><<<(unsigned)nq, 256, smem, st>>>(nq, parts, k_in, k_out, in_scores, in_labels, part_stride,
                                                                 q_stride, out_scores, out_labels, out_counts, P,
                                                                 dedupe ? 1 : 0, k_per_query);
    else
        merge_pairs_kernel<false><<<(unsigned)nq, 256, smem, st>>>(nq, parts, k_in, k_out, in_scores, in_labels, part_stride,
                                                                  q_stride, out_scores, out_labels, out_counts, P,
                                                                  dedupe ? 1 : 0, nullptr);
    return cudaGetLastError();
}

}  // namespace pyrope
