// flat_tc.cu — K1 on the 5th-gen tensor cores: batched exact FLAT scoring as a 3xTF32 split GEMM
// (tcgen05.mma kind::tf32, operands staged by TMA into 128B-swizzled shared memory, accumulators in
// TMEM) with the top-k selection fused into the epilogue, so the Q x N score matrix never exists.
//
// Replaces the scoring + heap loop of BruteForceVectorIndex.Search (BruteForceVectorIndex.cs:341-360)
// for a whole query batch, and — run over the centroid table — the coarse ranking of
// IvfFlatVectorIndex.cs:186-198 / IvfPqVectorIndex.cs:141-150.
//
//   D[q][n] = Qhi.Xhi + Qhi.Xlo + Qlo.Xhi      (hi = tf32(x) rounded to nearest, lo = x - hi, exact)
//   proxy score  s = scale[n] * D + bias[n]    (L2: 2*q.x - |x|^2 ; IP: q.x ; Cosine: q.x/|x| ;
//                                               tombstoned / out-of-range rows: bias = -inf)
// Tile: 128 queries (UMMA M, one TMEM lane each) x 256 base rows (UMMA N), K in 32-float chunks
// (one 128-byte swizzle atom), 2 shared-memory stages of 96 KiB, 2 TMEM accumulator buffers of 256
// columns.  Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator,
// warps 4-7 = epilogue (thread <-> query: tcgen05.ld its lane, compare against its private
// threshold, append survivors to its private queue in L2; a full queue is sorted by the whole warp).
// The k' = k + margin survivors per (query, split) are re-scored with exact fp32 arithmetic by
// flat_rescore_kernel, which also does the final ordering — reported distances never come from
// the tensor path.
//
// Long rows (d > 256, >= 65,536 rows: BASELINE config 4) take ONE product per K slice instead of three — on fp16
// copies of both operands (kind::f16) when the values fit, else on the tf32 hi copies — with a rigorous rounding
// band per query (tc_band_kernel) and a three-term pass behind that only runs if a queue overflowed; one-term
// passes use four 48 KiB stages and are launched in clusters of two CTAs that multicast the X chunks to each other.
#include <cuda.h>

#include <algorithm>

#include "common.cuh"
#include "exact_arith.cuh"
#include "kernels.h"

namespace pyrope {
namespace {

constexpr int BM = 128, BN = 256, BK = 32, STAGES = 2;
constexpr int TC_THREADS = 384;  // TMA, MMA, TMEM-alloc, spare + 4 epilogue warps (+ 4 more when the columns are halved)
constexpr int QH_BYTES = BM * BK * 4, XH_BYTES = BN * BK * 4;
constexpr int STAGE_BYTES = 2 * QH_BYTES + 2 * XH_BYTES;  // 96 KiB
constexpr int TMEM_COLS = 512;

// ---- PTX wrappers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One lane of a CONVERGED warp.  The single-thread roles (TMA producer, MMA issuer) must be entered through this and not
// through `lane == 0`: ptxas knows elect.sync yields exactly one lane and keeps descriptors in uniform registers, whereas
// under a plain divergent branch it wraps every UTCHMMA / UTMALDG in an ELECT + R2UR.BROADCAST + BRA.U.ANY loop over the
// "possibly several" active threads — measured 166 cycles of issue per tcgen05.mma against a 64-cycle tensor-pipe floor.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 28)) __trap();  // a broken pipeline must fault, not hang the GPU
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
// the same into the shared memory of every CTA of the cluster named in `mask` (same offset), completing bytes on each
// CTA's own barrier at the same offset
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
        : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// arrive on the barrier at this offset in every CTA of `mask` once the MMAs issued so far have retired
__device__ __forceinline__ void tc_commit_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
        : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
        : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// K-major operand tile in shared memory, 128-byte rows, SWIZZLE_128B, 8-row atoms of 1024 bytes
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);  // start address
    d |= (uint64_t)0 << 16;                    // leading byte offset (unused: one atom along K)
    d |= (uint64_t)(1024 >> 4) << 32;          // stride byte offset between 8-row atoms
    d |= (uint64_t)1 << 46;                    // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
    return d;
}
// kind::tf32, fp32 accumulate, A and B K-major, M = 128, N = 256
constexpr uint32_t kInstrDesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
// kind::f16, fp16 operands (format 0), fp32 accumulate: 16 elements per MMA, 64 per 128-byte chunk
constexpr uint32_t kInstrDescF16 = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
// one-term passes load one Q and one X chunk per stage (48 KiB): four stages fit where the three-term split holds two
constexpr int STAGES1 = 4, STAGE1_BYTES = QH_BYTES + XH_BYTES;
static_assert(STAGES1 * STAGE1_BYTES == STAGES * STAGE_BYTES, "both layouts fill the same shared memory");

struct TcParams {
    int64_t nq, n_scan;
    int dim, kprime, cap, splits;
    int64_t ntiles, tiles_per_split;
    const float* scale;  // [n] nullable (=1)
    const float* bias;   // [n] nullable (=0)
    uint64_t* queue;     // [splits][nq_pad][cap]
    int32_t* counts;     // [splits][nq_pad]
    int64_t nq_pad;
    // two-pass threshold (epilogue-bound shapes): pass A (gmax != null) only records, per query, the
    // maximum proxy score of every 32-row group; pass B starts every query at tau_init instead of -inf
    float uscale;        // metric with one scale for every row (L2: 2, IP: 1): skip the per-row scale loads
    int has_uscale;
    int one_term;        // D = Qhi.Xhi only (one product per K slice; the band / select step covers the error)
    int f16;             // one_term with fp16 operands behind map_qhi / map_xhi (kind::f16)
    // one_term, launched as clusters of two CTAs (neighbouring query tiles, same row range): each CTA fetches HALF of every X
    // chunk and multicasts it into both (map_xlo = the half-height X box), so a chunk costs 32 KiB of L2 -> SM traffic per
    // SM instead of 48.  qtiles_grid = query tiles rounded up to a whole number of clusters: the CTAs past the last real
    // tile are ghosts that only fetch and release.  (Measured on C4: 159 -> 147 ms per batch at 2 CTAs, no further gain at
    // 4; an L2 prefetch of the next tile's rows made it slower.  The kernel runs under the board's power cap - SM clock
    // ~1.1-1.45 GHz of 1.965 - so what counts is energy per MMA, not bytes in flight.)
    int cluster;         // CTAs per cluster (0: none, 2 or 4): each fetches 1/cluster of every X chunk
    int64_t qtiles_grid;
    float* gmax;         // [nq_pad][gstride]
    int64_t gstride;     // groups per query = ntiles * 8
    const float* tau_init;  // [nq_pad] nullable
    // pass B with ONE tf32 product: scores are off by at most band/2 from the exact proxy, so pruning keeps
    // everything within `band` of the k'-th best and the threshold trails it by `band`; a queue that cannot be
    // pruned below its capacity raises *overflow and the three-term kernel (run_if = overflow) redoes the batch
    const float* band;   // [nq_pad] nullable (null: three-term scores, exact pruning)
    int* overflow;       // nullable
    const int* run_if;   // nullable: the whole grid exits at once unless *run_if != 0
    // epilogue-bound shapes: 2 = eight epilogue warps, warps 8-11 take the upper half of every tile's columns and keep
    // their own queues (part index = split * halves + half); 1 = four epilogue warps (warps 8-11 idle)
    int halves;
};

__global__ void __launch_bounds__(TC_THREADS, 1)
flat_tc_kernel(const __grid_constant__ CUtensorMap map_qhi, const __grid_constant__ CUtensorMap map_qlo,
               const __grid_constant__ CUtensorMap map_xhi, const __grid_constant__ CUtensorMap map_xlo, TcParams p) {
    if (p.run_if && *p.run_if == 0) return;  // fallback pass of the one-term path: nothing overflowed
    extern __shared__ __align__(1024) uint8_t smem[];
    // layout: [stage0 | stage1 | barriers | tmem ptr | per epilogue warp: sbias[2][BN], sscale[2][BN]]
    uint8_t* stage_base = smem;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(bars + 16);
    float* sterms = reinterpret_cast<float*>(tmem_ptr_s + 4);  // [4 warps][bias 2*BN | scale 2*BN]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES1]);
    const uint32_t tfull0 = smem_u32(&bars[2 * STAGES1]), tempty0 = smem_u32(&bars[2 * STAGES1 + 2]);
    // stage ring: four 48 KiB stages (one Q chunk, one X chunk) for one-term passes, two 96 KiB stages (hi and lo of both)
    const uint32_t nsm = p.one_term ? STAGES1 - 1 : STAGES - 1, nsh = p.one_term ? 2 : 1;
    const uint32_t stage_bytes = p.one_term ? STAGE1_BYTES : STAGE_BYTES, xoff = p.one_term ? QH_BYTES : 2 * QH_BYTES;
    const int BKE = p.f16 ? 2 * BK : BK;  // elements per 128-byte K chunk

    const int64_t qtiles = (p.nq + BM - 1) / BM;
    const int64_t qtg = p.cluster ? p.qtiles_grid : qtiles;
    const int64_t qt = blockIdx.x % qtg, sp = blockIdx.x / qtg;
    const bool ghost = qt >= qtiles;
    uint32_t crank = 0;
    if (p.cluster) asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
    const uint16_t cmask = (uint16_t)((1u << p.cluster) - 1u);
    const int64_t t_begin = sp * p.tiles_per_split;
    const int64_t t_end = min(p.ntiles, t_begin + p.tiles_per_split);
    const int ntile = (int)max((int64_t)0, t_end - t_begin);
    const int KC = (p.dim + BKE - 1) / BKE;

    if (tid == 0) {
        for (int i = 0; i < STAGES1; ++i) { mbar_init(full0 + 8 * i, 1); mbar_init(empty0 + 8 * i, p.cluster ? p.cluster : 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(tfull0 + 8 * i, 1); mbar_init(tempty0 + 8 * i, 4 * p.halves); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_s)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (p.cluster) cluster_sync_all();  // the partner's barriers exist before anything is multicast at them
    const uint32_t tmem_base = *tmem_ptr_s;

    if (warp == 0) {
        // ================= TMA producer =================
        if (elect_one()) {
            uint32_t it = 0;
            if (p.cluster) {
                for (int ti = 0; ti < ntile; ++ti) {
                    const int n0 = (int)((t_begin + ti) * BN);
                    for (int kc = 0; kc < KC; ++kc, ++it) {
                        const uint32_t s = it & nsm, ph = (it >> nsh) & 1;
                        mbar_wait(empty0 + 8 * s, ph ^ 1);  // both CTAs have finished with the stage
                        const uint32_t sb = smem_u32(stage_base) + s * stage_bytes;
                        mbar_expect_tx(full0 + 8 * s, ghost ? XH_BYTES : stage_bytes);
                        if (!ghost) tma_load_2d(sb, &map_qhi, full0 + 8 * s, kc * BKE, (int)(qt * BM));
                        tma_load_2d_mc(sb + xoff + crank * (XH_BYTES / p.cluster), &map_xlo, full0 + 8 * s, kc * BKE,
                                       n0 + (int)crank * (BN / p.cluster), cmask);
                    }
                }
            } else
            for (int ti = 0; ti < ntile; ++ti) {
                const int n0 = (int)((t_begin + ti) * BN);
                for (int kc = 0; kc < KC; ++kc, ++it) {
                    const uint32_t s = it & nsm, ph = (it >> nsh) & 1;
                    mbar_wait(empty0 + 8 * s, ph ^ 1);
                    const uint32_t sb = smem_u32(stage_base) + s * stage_bytes;
                    mbar_expect_tx(full0 + 8 * s, stage_bytes);
                    tma_load_2d(sb, &map_qhi, full0 + 8 * s, kc * BKE, (int)(qt * BM));
                    tma_load_2d(sb + xoff, &map_xhi, full0 + 8 * s, kc * BKE, n0);
                    if (!p.one_term) {
                        tma_load_2d(sb + QH_BYTES, &map_qlo, full0 + 8 * s, kc * BK, (int)(qt * BM));
                        tma_load_2d(sb + 2 * QH_BYTES + XH_BYTES, &map_xlo, full0 + 8 * s, kc * BK, n0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (elect_one()) {
            uint32_t it = 0;
            if (ghost) {  // no queries here: take delivery of every stage and hand it back
                for (int64_t n = (int64_t)ntile * KC; n > 0; --n, ++it) {
                    const uint32_t s = it & nsm, ph = (it >> nsh) & 1;
                    mbar_wait(full0 + 8 * s, ph);
                    tc_commit_mc(empty0 + 8 * s, cmask);
                }
            } else
            for (int ti = 0; ti < ntile; ++ti) {
                const uint32_t buf = ti & 1, aph = (ti >> 1) & 1;
                mbar_wait(tempty0 + 8 * buf, aph ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * BN;
                for (int kc = 0; kc < KC; ++kc, ++it) {
                    const uint32_t s = it & nsm, ph = (it >> nsh) & 1;
                    mbar_wait(full0 + 8 * s, ph);
                    tc_fence_after();
                    const uint32_t sb = smem_u32(stage_base) + s * stage_bytes;
                    const uint64_t qhi = make_sw128_desc(sb), qlo = make_sw128_desc(sb + QH_BYTES);
                    const uint64_t xhi = make_sw128_desc(sb + xoff), xlo = make_sw128_desc(sb + 2 * QH_BYTES + XH_BYTES);
#pragma unroll
                    for (int k4 = 0; k4 < BK / 8; ++k4) {
                        const uint64_t adv = (uint64_t)(k4 * 2);  // 8 floats = 32 bytes = 2 x 16-byte units
                        if (p.f16) {
                            tc_mma_f16(d_tmem, qhi + adv, xhi + adv, kInstrDescF16, (kc | k4) != 0);
                        } else if (p.one_term) {
                            tc_mma_tf32(d_tmem, qhi + adv, xhi + adv, kInstrDesc, (kc | k4) != 0);
                        } else {
                            tc_mma_tf32(d_tmem, qlo + adv, xhi + adv, kInstrDesc, (kc | k4) != 0);
                            tc_mma_tf32(d_tmem, qhi + adv, xlo + adv, kInstrDesc, 1);
                            tc_mma_tf32(d_tmem, qhi + adv, xhi + adv, kInstrDesc, 1);
                        }
                    }
                    // frees the shared-memory stage when these MMAs retire (in both CTAs of a cluster: the partner writes here too)
                    if (p.cluster) tc_commit_mc(empty0 + 8 * s, cmask); else tc_commit(empty0 + 8 * s);
                }
                tc_commit(tfull0 + 8 * buf);    // accumulator tile complete
            }
        }
    } else if (warp >= 4 && warp < 4 + 4 * p.halves && !ghost) {
        // ================= epilogue: thread <-> query (x column half) =================
        const int ew = (warp - 4) & 3;                 // TMEM lane quarter
        const int hf = (warp - 4) >> 2;                // column half of every tile this warp reads
        const int HN = BN / p.halves;                  // columns per epilogue warp and tile
        const int CH = HN / 32;                        // 32-column chunks of them
        const int et = ew * 32 + lane;                 // 0..127
        const int64_t gq = qt * BM + et;
        const bool qvalid = gq < p.nq;
        const int64_t part = sp * p.halves + hf;
        uint64_t* myq = p.queue + (part * p.nq_pad + (qt * BM + et)) * p.cap;
        float* sbias = sterms + (warp - 4) * (4 * HN);   // private to this warp: the epilogue warps never wait
        float* sscale = sbias + 2 * HN;                 // for one another, only for the MMA warp (mbarriers)
        int cnt = 0;
        const bool gmode = p.gmax != nullptr;
        float tau = (!gmode && p.tau_init && qvalid) ? __ldg(p.tau_init + gq) : -INFINITY;
        const float band = (!gmode && p.band && qvalid) ? __ldg(p.band + gq) : 0.f;
        const int cap = p.cap, kprime = p.kprime;

        // Keep the k' best keys of lane l's queue (in L2), whole warp cooperating, queue held in
        // registers: a bisection on the 32-bit ordered score finds the k'-th largest score T, keys above
        // T (and as many keys equal to T as still fit) are compacted back; no sort, no shared memory.
        auto prune_lane = [&](int l) {
            uint64_t* src = reinterpret_cast<uint64_t*>(__shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)myq, l));
            const int c = __shfl_sync(0xffffffffu, cnt, l);
            if (c <= kprime) return;  // warp-uniform
            constexpr int U = 16;     // cap <= 512
            const int cu = (c + 31) >> 5;  // occupied registers per lane (warp-uniform)
            uint64_t e[U];
            uint32_t o[U];                 // ordered scores; empty slots hold 0 (below every valid score)
            uint32_t lo = 0xffffffffu, hi = 0u;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = u * 32 + lane;
                e[u] = (u < cu && i < c) ? __ldcg(src + i) : 0ull;
                o[u] = (uint32_t)(e[u] >> 32);
                if (e[u]) { lo = min(lo, o[u]); hi = max(hi, o[u]); }
            }
            lo = __reduce_min_sync(0xffffffffu, lo);
            hi = __reduce_max_sync(0xffffffffu, hi);
            while (lo < hi) {  // largest T with count(ord >= T) >= k'   (mid > lo >= 1: empty slots never count)
                const uint32_t mid = lo + ((hi - lo + 1u) >> 1);
                int n = 0;
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (u < cu) n += (o[u] >= mid);
                n = __reduce_add_sync(0xffffffffu, n);
                if (n >= kprime) lo = mid; else hi = mid - 1u;
            }
            uint32_t T = lo;
            const float bl = __shfl_sync(0xffffffffu, band, l);
            int quota, out = 0;
            if (bl > 0.f) {
                // approximate scores: everything within the band below the k'-th best may still beat it once
                // re-scored, so it all stays (ties included: no quota)
                T = score_to_ord(ord_to_score(lo) - bl);
                int nk = 0;
#pragma unroll
                for (int u = 0; u < U; ++u) nk += (e[u] != 0ull && o[u] >= T);
                nk = __reduce_add_sync(0xffffffffu, nk);
                if (nk > cap - 64) {  // cannot shrink: flag the batch for the exact fallback, keep going with exactly k'
                    if (lane == 0 && p.overflow) atomicExch(p.overflow, 1);
                    T = lo;
                    quota = -1;
                } else {
                    T = T > 0u ? T - 1u : 0u;  // keep o >= threshold  <=>  o > T
                    quota = 0;
                }
            } else {
                quota = -1;
            }
            if (quota < 0) {
                int ngt = 0;
#pragma unroll
                for (int u = 0; u < U; ++u) ngt += (o[u] > T);
                ngt = __reduce_add_sync(0xffffffffu, ngt);
                quota = kprime - ngt;  // ties at T still admitted
            }
            const unsigned below = (1u << lane) - 1u;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (u >= cu) break;
                const bool gt = o[u] > T, eq = e[u] != 0ull && o[u] == T;
                const unsigned meq = __ballot_sync(0xffffffffu, eq);
                const bool take_eq = eq && (int)__popc(meq & below) < quota;
                quota -= min(quota, (int)__popc(meq));
                const unsigned mk = __ballot_sync(0xffffffffu, gt || take_eq);
                if (gt || take_eq) __stcg(src + out + __popc(mk & below), e[u]);
                out += __popc(mk);
            }
            if (lane == l) {
                cnt = out;  // == k' (more with a band)
                tau = ord_to_score(T);
            }
            __syncwarp();
        };

        // per-row scale/bias of a tile (8 columns per lane, private copy per warp), fetched ONE TILE AHEAD so
        // the L2 round trip hides behind the current tile's epilogue
        float nb[BN / 32], ns[BN / 32];
        auto load_terms = [&](int ti) {
            const int64_t n0 = (t_begin + ti) * BN + hf * HN;
#pragma unroll
            for (int u = 0; u < BN / 32; ++u) {
                if (u >= CH) break;
                const int64_t pos = n0 + lane + u * 32;
                nb[u] = -INFINITY; ns[u] = 0.f;
                if (pos < p.n_scan) {
                    nb[u] = p.bias ? __ldg(p.bias + pos) : 0.f;
                    ns[u] = (p.scale && !p.has_uscale) ? __ldg(p.scale + pos) : 1.f;
                }
            }
        };
        auto store_terms = [&](uint32_t buf) {
#pragma unroll
            for (int u = 0; u < BN / 32; ++u) {
                if (u >= CH) break;
                sbias[buf * HN + lane + u * 32] = nb[u];
                sscale[buf * HN + lane + u * 32] = ns[u];
            }
            __syncwarp();
        };
        if (ntile > 0) { load_terms(0); store_terms(0); }
        for (int ti = 0; ti < ntile; ++ti) {
            const uint32_t buf = ti & 1, aph = (ti >> 1) & 1;
            const int64_t n0 = (t_begin + ti) * BN;
            if (ti + 1 < ntile) load_terms(ti + 1);  // consumed after this tile
            mbar_wait(tfull0 + 8 * buf, aph);
            tc_fence_after();
            const uint32_t taddr0 = tmem_base + ((uint32_t)(ew * 32) << 16) + buf * BN;
#pragma unroll 1
            for (int c = hf * CH; c < hf * CH + CH; ++c) {
                float v[32];
                tc_ld32(taddr0 + c * 32, v);
                if (qvalid) {  // proxy scores, in place: v = D * scale + bias (row terms read 4 columns at a time)
                    const float4* b4 = reinterpret_cast<const float4*>(sbias + buf * HN + (c - hf * CH) * 32);
                    const float4* s4 = reinterpret_cast<const float4*>(sscale + buf * HN + (c - hf * CH) * 32);
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4) {
                        const float4 bb = b4[j4];
                        float4 ss = make_float4(p.uscale, p.uscale, p.uscale, p.uscale);
                        if (!p.has_uscale) ss = s4[j4];
                        v[4 * j4 + 0] = fmaf(v[4 * j4 + 0], ss.x, bb.x);
                        v[4 * j4 + 1] = fmaf(v[4 * j4 + 1], ss.y, bb.y);
                        v[4 * j4 + 2] = fmaf(v[4 * j4 + 2], ss.z, bb.z);
                        v[4 * j4 + 3] = fmaf(v[4 * j4 + 3], ss.w, bb.w);
                    }
                }
                if (qvalid && gmode) {
                    float mx = -INFINITY;
#pragma unroll
                    for (int j = 0; j < 32; ++j) mx = fmaxf(mx, v[j]);
                    p.gmax[gq * p.gstride + (t_begin + ti) * (BN / 32) + c] = mx;
                } else if (qvalid) {
                    // common case after warm-up: no proxy score of an 8-column group beats the threshold; the
                    // element-wise test (divergent: lanes are different queries) runs only for groups with a hit
                    float gm[4];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        gm[g] = -INFINITY;
#pragma unroll
                        for (int j = g * 8; j < g * 8 + 8; ++j) gm[g] = fmaxf(gm[g], v[j]);
                    }
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        if (gm[g] > tau) {
#pragma unroll
                            for (int j = g * 8; j < g * 8 + 8; ++j) {
                                if (v[j] > tau) {
                                    __stcg(myq + cnt, make_key(v[j], (uint32_t)(n0 + c * 32 + j)));
                                    ++cnt;
                                }
                            }
                        }
                    }
                }
                unsigned full = gmode ? 0u : __ballot_sync(0xffffffffu, cnt > cap - 32);
                while (full) {
                    const int l = __ffs(full) - 1;
                    full &= full - 1;
                    prune_lane(l);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty0 + 8 * buf);
            if (ti + 1 < ntile) store_terms(buf ^ 1);
        }
        // final: leave the best k' (unordered) in place, publish the counts
        if (!gmode) {
            for (int l = 0; l < 32; ++l) prune_lane(l);
            p.counts[part * p.nq_pad + qt * BM + et] = qvalid ? cnt : 0;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (p.cluster) cluster_sync_all();  // the partner may still be multicasting data and arrivals into this CTA
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// ---- two-pass threshold: the k'-th largest group maximum bounds the k'-th best score from below -------
// (each of the k' best groups holds at least one row scoring >= its maximum).  One warp per query.
// When pass A ran with ONE tf32 product (hi.hi only) its scores differ from the 3-term proxy by at most
// eps_q = 2^-10 (1 + 2^-7) |q| max_r(|scale_r| |x_r|)  (each operand rounded to 11 significant bits, Cauchy-
// Schwarz), so tau is lowered by eps_q (+ the same again for the 3-term side's own rounding, generously).
__global__ void __launch_bounds__(128) tc_gmax_select_kernel(const float* __restrict__ gmax, int64_t gstride, int ngroups,
                                                            int64_t nq, int kprime, float* tau_out,
                                                            const float* __restrict__ Q, int dim,
                                                            const float* __restrict__ amax, float* band_out, int* overflow) {
    const int64_t q = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0 && overflow) *overflow = 0;
    if (q >= nq) return;
    float band = 0.f;
    const float* g = gmax + q * gstride;
    float tau = -INFINITY;
    if (ngroups > kprime) {
        constexpr int R = 64;  // register-resident up to 2048 groups, re-read from L1/L2 beyond
        const bool in_regs = ngroups <= R * 32;
        uint32_t o[R];
        uint32_t lo = 0xffffffffu, hi = 0u;
        if (in_regs) {
#pragma unroll
            for (int u = 0; u < R; ++u) {
                const int i = u * 32 + lane;
                o[u] = i < ngroups ? score_to_ord(__ldg(g + i)) : 0u;
                if (i < ngroups) { lo = min(lo, o[u]); hi = max(hi, o[u]); }
            }
        } else {
            for (int i = lane; i < ngroups; i += 32) {
                const uint32_t v = score_to_ord(__ldg(g + i));
                lo = min(lo, v);
                hi = max(hi, v);
            }
        }
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        while (lo < hi) {  // largest T with count(ord >= T) >= k'   (mid > lo >= 1: padding zeros never count)
            const uint32_t mid = lo + ((hi - lo + 1u) >> 1);
            int n = 0;
            if (in_regs) {
#pragma unroll
                for (int u = 0; u < R; ++u) n += o[u] >= mid;
            } else {
                for (int i = lane; i < ngroups; i += 32) n += score_to_ord(__ldg(g + i)) >= mid;
            }
            n = __reduce_add_sync(0xffffffffu, n);
            if (n >= kprime) lo = mid; else hi = mid - 1u;
        }
        tau = lo > 1u ? ord_to_score(lo - 1u) : -INFINITY;  // pass B accepts s > tau, i.e. s >= value(T)
        if (amax) {
            float qq = 0.f;
            for (int d = lane; d < dim; d += 32) { const float v = __ldg(Q + q * dim + d); qq = fmaf(v, v, qq); }
            qq = warp_sum(qq);
            const float eps = 2.f * 9.85e-4f * sqrtf(qq) * __ldg(amax);  // 2 x 2^-10 (1 + 2^-7) |q| A
            tau -= eps + 1e-6f * fabsf(tau);
            // a one-term pass B sees the same scores as pass A: a row of the true top k' scores at least
            // (k'-th group maximum) - eps there, which is this tau; its pruning band is the same 2 x eps_q
            band = eps + 1e-6f * fabsf(tau);
        }
    }
    if (lane == 0) {
        tau_out[q] = tau;
        if (band_out) band_out[q] = band;
    }
}

// ---- single one-TF32 pass (long K: the FLAT scan of BASELINE config 4): no pass A, every query starts cold and prunes
// with the rounding band of the one-term product, eps_q = 2 x 2^-10 (1 + 2^-7) |q| max_r(|scale_r| |x_r|) (see above).
// fp16 operands: + the absolute error of components below 2^-14 (under = 2^-24 sqrt(d), smax = |scale|); a query with a
// component beyond the fp16 range gets an infinite band - its queue overflows and the three-term pass redoes the batch.
__global__ void __launch_bounds__(128) tc_band_kernel(const float* __restrict__ Q, int dim, int64_t nq, const float* __restrict__ amax,
                                                     float* band_out, int* overflow, float under, float smax,
                                                     const uint8_t* __restrict__ qbad) {
    const int64_t q = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) *overflow = 0;
    if (q >= nq) return;
    float qq = 0.f;
    for (int d = lane; d < dim; d += 32) { const float v = __ldg(Q + q * dim + d); qq = fmaf(v, v, qq); }
    qq = warp_sum(qq);
    if (lane == 0) {
        const float A = __ldg(amax), qn = sqrtf(qq);
        float b = 2.f * (9.85e-4f * qn * A + under * (smax * qn + A)) * 1.0001f + 1e-30f;
        if (qbad && qbad[q]) b = INFINITY;
        band_out[q] = b;
    }
}

// ---- exact fp32 re-score of the survivors + final ordering -------------------------------------
struct RescoreParams {
    const float* Q; int64_t nq; int dim;
    const float* X; const float* xnorm; const float* qnorm; const int64_t* labels;
    int metric, k, cap, splits;
    const uint64_t* queue; const int32_t* counts; int64_t nq_pad;
    int arith;  // 1: VectorMath.*Unsafe order (BruteForceVectorIndex.cs:350-356), 2: VectorMath.L2Squared / DotProduct order (IVF)
    PairOut out;
};

// The reference's evaluation orders, warp-cooperative, separate multiply and add (exact_arith.cuh conventions).
// a1 = L2SquaredUnsafe / DotProductUnsafe (VectorMath.cs:128-253): four 8-lane accumulators over 32-element blocks =
// 32 independent running sums, one per lane (coalesced 128-byte loads); final = ((a1 + a2) + a3) + a4 per lane j, then
// the pairwise horizontal sum; a separate accumulator for 1-3 leftover 8-blocks; scalar tail.  One candidate per warp.
template <int OP>
__device__ __forceinline__ float a1_eval_warp(const float* q, const float* __restrict__ x, int n, int lane) {
    int i = 0;
    float sum = 0.f;
    if (n >= 32) {
        float acc = 0.f;
        for (; i <= n - 32; i += 32) acc = __fadd_rn(acc, exact::term<OP>(q[i + lane], __ldg(x + i + lane)));
        const int j = lane & 7;
        const float v1 = __shfl_sync(0xffffffffu, acc, j), v2 = __shfl_sync(0xffffffffu, acc, 8 + j);
        const float v3 = __shfl_sync(0xffffffffu, acc, 16 + j), v4 = __shfl_sync(0xffffffffu, acc, 24 + j);
        float fin = __fadd_rn(__fadd_rn(__fadd_rn(v1, v2), v3), v4);
        fin = __fadd_rn(fin, __shfl_xor_sync(0xffffffffu, fin, 1));
        fin = __fadd_rn(fin, __shfl_xor_sync(0xffffffffu, fin, 2));
        fin = __fadd_rn(fin, __shfl_xor_sync(0xffffffffu, fin, 4));
        sum = __fadd_rn(sum, fin);
    }
    if (i <= n - 8) {
        float acc = 0.f;
        for (; i <= n - 8; i += 8)
            if (lane < 8) acc = __fadd_rn(acc, exact::term<OP>(q[i + lane], __ldg(x + i + lane)));
        acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, 1));
        acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, 2));
        acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, 4));
        sum = __fadd_rn(sum, __shfl_sync(0xffffffffu, acc, 0));
    }
    for (; i < n; ++i) sum = __fadd_rn(sum, exact::term<OP>(q[i], __ldg(x + i)));
    return sum;
}
// a2 = L2Squared / DotProduct (VectorMath.cs:8-70): one 8-lane accumulator stepping 8 elements.  Eight consecutive
// lanes (j = lane & 7) share a candidate: four candidates per warp.
template <int OP>
__device__ __forceinline__ float a2_eval_oct(const float* q, const float* __restrict__ x, int n, int j) {
    int i = 0;
    float sum = 0.f;
    if (n >= 8) {
        float acc = 0.f;
        for (; i <= n - 8; i += 8) acc = __fadd_rn(acc, exact::term<OP>(q[i + j], __ldg(x + i + j)));
        acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, 1));
        acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, 2));
        acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, 4));
        sum = __fadd_rn(sum, acc);
    }
    for (; i < n; ++i) sum = __fadd_rn(sum, exact::term<OP>(q[i], __ldg(x + i)));
    return sum;
}

// The survivors of a query are spread over `splits` queues; they pass through a window of P keys in shared memory:
// load up to P - (kept so far), score the new ones exactly, sort, keep the best k, repeat.  P >= 2k and P covers the
// usual total, so almost every query takes one round; only a query whose queues hold far more than expected (a band
// full of near-ties) takes several.
__global__ void __launch_bounds__(256) flat_rescore_kernel(RescoreParams p, int P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem_raw);  // [P]
    __shared__ int s_total;
    __shared__ int s_off[65];
    const int64_t q = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        int t = 0;
        for (int s = 0; s < p.splits; ++s) {
            s_off[s] = t;
            t += p.counts[(int64_t)s * p.nq_pad + q];
        }
        s_off[p.splits] = t;
        s_total = t;
    }
    __syncthreads();
    const int total = s_total;
    float* qv = reinterpret_cast<float*>(keys + P);  // the query, staged once
    for (int d = tid; d < p.dim; d += blockDim.x) qv[d] = p.Q[q * p.dim + d];
    const float qn = p.metric == kCosine ? p.qnorm[q] : 0.f;
    // survivors are scored in the REFERENCE's arithmetic: what is reported (and ranked) is the oracle's value bit for bit
    const int cpw = p.arith == 1 ? 1 : 4;       // candidates per warp and pass
    const int sub = p.arith == 1 ? 0 : lane >> 3;
    int kept = 0, off = 0, sorted_n = 0;
    do {
        const int n_new = min(total - off, P - kept);
        // gather: flat candidate index g -> (split, position) through the prefix sums
        for (int i = tid; i < n_new; i += blockDim.x) {
            const int g = off + i;
            int sidx = 0;
            while (sidx + 1 < p.splits && s_off[sidx + 1] <= g) ++sidx;
            keys[kept + i] = __ldcg(p.queue + ((int64_t)sidx * p.nq_pad + q) * p.cap + (g - s_off[sidx]));
        }
        __syncthreads();
        for (int i0 = kept + warp * cpw; i0 < kept + n_new; i0 += (blockDim.x >> 5) * cpw) {
            const int i = i0 + sub;
            const bool on = i < kept + n_new;
            const uint32_t pos = on ? key_pos(keys[i]) : key_pos(keys[i0]);  // idle lanes shadow a live candidate (shuffles stay uniform)
            const float* x = p.X + (int64_t)pos * p.dim;
            float a;
            if (p.arith == 1) a = p.metric == kL2 ? a1_eval_warp<0>(qv, x, p.dim, lane) : a1_eval_warp<1>(qv, x, p.dim, lane);
            else a = p.metric == kL2 ? a2_eval_oct<0>(qv, x, p.dim, lane & 7) : a2_eval_oct<1>(qv, x, p.dim, lane & 7);
            if (on && (p.arith == 1 ? lane == 0 : (lane & 7) == 0)) {
                float score;
                if (p.metric == kL2) score = -a;
                else if (p.metric == kIP) score = a;
                else {
                    const float xn = p.xnorm[pos];
                    score = (qn < 1e-6f || xn < 1e-6f) ? 0.f : __fdiv_rn(a, __fmul_rn(qn, xn));
                }
                keys[i] = make_key(score, pos);
            }
        }
        const int n = kept + n_new;
        const int P2 = next_pow2(max(n, 2));  // sort only as much as there is (block-uniform)
        for (int i = n + tid; i < P2; i += blockDim.x) keys[i] = 0ull;
        __syncthreads();
        bitonic_sort_desc<false>(keys, P2, tid, blockDim.x);
        off += n_new;
        kept = min(n, p.k);
        sorted_n = n;
    } while (off < total);
    const int have = min(sorted_n, total);
    const int64_t ob = (q * p.out.parts_total + p.out.part_base) * (int64_t)p.k;
    for (int i = tid; i < p.k; i += blockDim.x) {
        uint64_t key = (i < have) ? keys[i] : 0ull;
        if (key) {
            uint32_t pos = key_pos(key);
            p.out.scores[ob + i] = key_score(key);
            p.out.labels[ob + i] = p.labels ? p.labels[pos] : (int64_t)pos;
        } else {
            p.out.scores[ob + i] = 0.f;
            p.out.labels[ob + i] = -1;
        }
    }
}

// ---- operand preparation -----------------------------------------------------------------------
__global__ void tc_split_kernel(const float* __restrict__ X, int64_t n_elems, float* __restrict__ hi, float* __restrict__ lo) {
    int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < n_elems) {
        float4 x = __ldg(reinterpret_cast<const float4*>(X + i));
        float4 h, l;
        uint32_t t;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.x)); h.x = __uint_as_float(t);
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.y)); h.y = __uint_as_float(t);
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.z)); h.z = __uint_as_float(t);
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.w)); h.w = __uint_as_float(t);
        l.x = x.x - h.x; l.y = x.y - h.y; l.z = x.z - h.z; l.w = x.w - h.w;
        *reinterpret_cast<float4*>(hi + i) = h;
        *reinterpret_cast<float4*>(lo + i) = l;
    } else {
        for (; i < n_elems; ++i) {
            uint32_t t;
            float x = X[i];
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x));
            float h = __uint_as_float(t);
            hi[i] = h;
            lo[i] = x - h;
        }
    }
}

// one warp per row: scale/bias of the proxy score.  norms (cosine, may be null): the exact row norms of the re-score
__global__ void tc_rowterms_kernel(const float* __restrict__ X, int64_t n, int dim, int metric,
                                   const uint8_t* __restrict__ dead, const float* __restrict__ norms, float* scale,
                                   float* bias) {
    int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (r >= n) return;
    float a = 0.f;
    if (metric != kIP) {
        const float* x = X + r * dim;
        for (int d = lane; d < dim; d += 32) { float v = __ldg(x + d); a = fmaf(v, v, a); }
        a = warp_sum(a);
    }
    if (lane == 0) {
        float sc = 1.f, b = 0.f;
        if (metric == kL2) { sc = 2.f; b = -a; }
        else if (metric == kCosine) {
            // zero or not is decided on the exact norm, as the re-score and the reference (VectorMath.cs) decide it: this
            // lane-strided sum can land on the other side of 1e-6, and a crowd of rows that score 0 would then push the
            // scoring rows out of the candidates (or a scoring row would be dropped)
            const float nrm = sqrtf(a), cut = norms ? norms[r] : nrm;
            sc = (cut < 1e-6f || nrm == 0.f) ? 0.f : 1.f / nrm;
        }
        if (dead && dead[r]) b = -INFINITY;
        scale[r] = sc;
        bias[r] = b;
    }
}

// A = max over rows of |scale_r| * |x_r|  (float bits are order-preserving for non-negative values)
__global__ void tc_amax_kernel(const float* __restrict__ X, int64_t n, int dim, const float* __restrict__ scale, float* amax) {
    int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (r >= n) return;
    float a = 0.f;
    for (int d = lane; d < dim; d += 32) { float v = __ldg(X + r * dim + d); a = fmaf(v, v, a); }
    a = warp_sum(a);
    if (lane == 0) atomicMax(reinterpret_cast<unsigned int*>(amax), __float_as_uint(fabsf(scale ? scale[r] : 1.f) * sqrtf(a)));
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

bool make_map(CUtensorMap* m, const void* base, int64_t rows, int dim, int box_rows, bool f16 = false) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return false;
    cuuint64_t gdim[2] = {(cuuint64_t)dim, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)dim * (f16 ? 2 : 4)};
    cuuint32_t box[2] = {(cuuint32_t)(f16 ? 2 * BK : BK), (cuuint32_t)box_rows};  // 128 bytes wide either way
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

}  // namespace

// ---- public launchers ----------------------------------------------------------------------------
int flat_tc_margin(int k) { return k < 64 ? 16 : 32; }
bool flat_tc_supported(int dim, int k) { return dim % 4 == 0 && dim >= 8 && k >= 1 && k + flat_tc_margin(k) <= 224; }
// queue capacity per (split, query): a prune (register-resident bisection select by the whole warp) fires
// when fewer than 32 slots are left and keeps k'; the headroom cap - 32 - k' is the number of candidates
// accepted between two prunes.
int flat_tc_parts_per_split(const FlatTcParams& a) { return (a.gmax_ws && a.tau_ws) ? 2 : 1; }
int flat_tc_cap(int kprime) { return std::min(512, std::max(128, next_pow2(4 * kprime + 32))); }
int64_t flat_tc_nq_pad(int64_t nq) { return (nq + BM - 1) / BM * BM; }

// long K (many MMAs per tile): the scan is bound by operand traffic and MMAs, not by the epilogue — one TF32 term with
// band pruning instead of the three-term split
bool flat_tc_oneterm(int dim, int64_t n_scan, int kprime) {
    return dim > 256 && n_scan >= 65536 && kprime <= 224 && !getenv("PYROPE_TC_3X");
}
bool flat_tc_twopass(int dim, int64_t n_scan, int kprime) {
    // epilogue-bound regime only: short K (few MMAs per tile), a long stream and a wide k'
    return dim <= 256 && n_scan >= 16384 && kprime >= 32 && !getenv("PYROPE_TC_ONEPASS");
}
size_t flat_tc_gmax_floats(int64_t nq, int64_t n_scan) {
    return (size_t)flat_tc_nq_pad(nq) * (size_t)((n_scan + BN - 1) / BN) * (BN / 32);
}

// splits when every query already has a threshold (two-pass) or no per-split state at all (pass A): only
// wave quantisation and a small fixed cost per CTA matter
static int pick_splits_seeded(int64_t nq, int64_t n_scan, int num_sms, int64_t smax_extra) {
    const int64_t qtiles = (nq + BM - 1) / BM;
    const int64_t ntiles = std::max<int64_t>(1, (n_scan + BN - 1) / BN);
    const int64_t smax = std::min<int64_t>(std::min<int64_t>(ntiles, 32), smax_extra);
    int best = 1;
    double best_cost = 1e300;
    for (int64_t s = 1; s <= smax; ++s) {
        const int64_t tps = (ntiles + s - 1) / s;
        if (s > 1 && tps < 8) break;
        const int64_t waves = (qtiles * s + num_sms - 1) / num_sms;
        const double cost = (double)waves * ((double)tps + 2.0);
        if (cost < best_cost * 0.98) { best_cost = cost; best = (int)s; }
    }
    return best;
}

int flat_tc_pick_splits_seeded(int64_t nq, int64_t n_scan, int kprime, int num_sms) {
    // two column halves per split, up to cap entries each within the band: the re-score holds them all in shared
    // memory (16,384 keys = 128 KiB), so at most 16 splits
    return pick_splits_seeded(nq, n_scan, num_sms, std::min<int64_t>(16, std::max<int64_t>(1, 4096 / kprime)));
}

int flat_tc_pick_splits(int64_t nq, int64_t n_scan, int kprime, int num_sms) {

    // One CTA owns a 128-query tile and streams n-tiles of 256 rows.  Splitting the row range fills idle
    // SMs when there are few query tiles, but every split starts with no threshold (its first ~2 tiles
    // are accepted wholesale) and hands k' more candidates per query to the exact re-score, so a split
    // must keep a long stream: cost model = waves x (tiles per split + a fixed per-split charge).
    const int64_t qtiles = (nq + BM - 1) / BM;
    const int64_t ntiles = std::max<int64_t>(1, (n_scan + BN - 1) / BN);
    const int64_t smax = std::min<int64_t>(std::min<int64_t>(ntiles, 32), std::max<int64_t>(1, 4096 / kprime));
    const double per_split = 4.0 + kprime / 8.0;  // tiles' worth of selection + re-score work
    int best = 1;
    double best_cost = 1e300;
    for (int64_t s = 1; s <= smax; ++s) {
        const int64_t tps = (ntiles + s - 1) / s;
        if (s > 1 && tps < 16) break;
        const int64_t waves = (qtiles * s + num_sms - 1) / num_sms;
        const double cost = (double)waves * ((double)tps + per_split);
        if (cost < best_cost * 0.97) { best_cost = cost; best = (int)s; }  // prefer fewer splits on near ties
    }
    return best;
}

cudaError_t launch_tc_prepare(const float* X, int64_t n, int dim, int metric, const uint8_t* dead, float* hi, float* lo,
                              float* scale, float* bias, int64_t from_row, cudaStream_t st, const float* norms) {
    if (n <= from_row) return cudaSuccess;
    const int64_t rows = n - from_row;
    const int64_t ne = rows * dim;
    tc_split_kernel<<<(unsigned)((ne / 4 + 256) / 256), 256, 0, st>>>(X + from_row * dim, ne, hi + from_row * dim, lo + from_row * dim);
    if (scale && bias)
        tc_rowterms_kernel<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, st>>>(X + from_row * dim, rows, dim, metric,
                                                                            dead ? dead + from_row : nullptr,
                                                                            norms ? norms + from_row : nullptr, scale + from_row,
                                                                            bias + from_row);
    return cudaGetLastError();
}

cudaError_t launch_tc_amax(const float* X, int64_t n, int dim, const float* scale, float* amax, int64_t from_row,
                           cudaStream_t st) {
    if (n <= from_row) return cudaSuccess;
    const int64_t rows = n - from_row;
    tc_amax_kernel<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, st>>>(X + from_row * dim, rows, dim,
                                                                        scale ? scale + from_row : nullptr, amax);
    return cudaGetLastError();
}

cudaError_t launch_tc_rowterms(const float* X, int64_t n, int dim, int metric, const uint8_t* dead, float* scale, float* bias,
                               cudaStream_t st, const float* norms) {
    if (n <= 0) return cudaSuccess;
    tc_rowterms_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, st>>>(X, n, dim, metric, dead, norms, scale, bias);
    return cudaGetLastError();
}

// mode: 0 = three-term scores; 1 = one-term pass B (band pruning, raises the overflow flag); 2 = three-term fallback that
// runs only if the flag was raised
static cudaError_t launch_flat_tc_pass(const FlatTcParams& a, int splits, float* gmax, const float* tau_init, cudaStream_t st,
                                       int mode = 0);
// the two-pass path is the epilogue-bound regime: eight epilogue warps, two column halves per tile, each with its own
// queues, so a (split, query) pair owns flat_tc_parts_per_split() parts of queue / counts
// one-term pass B: tau_ws holds [tau | band | overflow flag]
static bool one_term_b(const FlatTcParams& a) { return a.gmax_ws && a.tau_ws && a.amax && !getenv("PYROPE_TC_PASSB_3X"); }

cudaError_t launch_flat_tc_select(const FlatTcParams& a, cudaStream_t st) {
    if (a.nq <= 0) return cudaSuccess;
    if (!a.gmax_ws && a.tau_ws && a.amax) {
        // ONE one-TF32 pass with band pruning (a third of the MMAs and half the operand traffic of the 3xTF32 split);
        // a queue that cannot be pruned below its capacity raises the flag and the three-term pass behind redoes the batch
        const int64_t nq_pad = flat_tc_nq_pad(a.nq);
        const bool f16 = a.Q16 && a.X16;
        tc_band_kernel<<<(unsigned)((a.nq + 3) / 4), 128, 0, st>>>(a.Q, a.dim, a.nq, a.amax, a.tau_ws + nq_pad,
                                                                   reinterpret_cast<int*>(a.tau_ws + 2 * nq_pad),
                                                                   f16 ? 5.97e-8f * sqrtf((float)a.dim) : 0.f,
                                                                   a.metric == kL2 ? 2.f : 1.f, f16 ? a.qbad : nullptr);
        cudaError_t e = launch_flat_tc_pass(a, a.splits, nullptr, nullptr, st, 1);
        if (e != cudaSuccess) return e;
        return launch_flat_tc_pass(a, a.splits, nullptr, nullptr, st, 2);
    }
    if (a.gmax_ws && a.tau_ws) {  // two-pass threshold
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaError_t e = launch_flat_tc_pass(a, pick_splits_seeded(a.nq, a.n_scan, sms, 32), a.gmax_ws, nullptr, st);
        if (e != cudaSuccess) return e;
        const int64_t ntiles = (a.n_scan + BN - 1) / BN;
        const int64_t nq_pad = flat_tc_nq_pad(a.nq);
        const bool ot = one_term_b(a);
        tc_gmax_select_kernel<<<(unsigned)((a.nq + 3) / 4), 128, 0, st>>>(a.gmax_ws, ntiles * (BN / 32), (int)(ntiles * (BN / 32)),
                                                                           a.nq, a.kprime, a.tau_ws, a.Q, a.dim, a.amax,
                                                                           ot ? a.tau_ws + nq_pad : nullptr,
                                                                           ot ? reinterpret_cast<int*>(a.tau_ws + 2 * nq_pad) : nullptr);
        if (!ot) return launch_flat_tc_pass(a, a.splits, nullptr, a.tau_ws, st);
        e = launch_flat_tc_pass(a, a.splits, nullptr, a.tau_ws, st, 1);
        if (e != cudaSuccess) return e;
        return launch_flat_tc_pass(a, a.splits, nullptr, a.tau_ws, st, 2);
    }
    return launch_flat_tc_pass(a, a.splits, nullptr, nullptr, st);
}

static cudaError_t launch_flat_tc_pass(const FlatTcParams& a, int splits, float* gmax, const float* tau_init, cudaStream_t st,
                                       int mode) {
    CUtensorMap mqh, mql, mxh, mxl;
    const bool f16 = mode == 1 && !gmax && a.Q16 && a.X16;  // the single one-term pass on fp16 copies
    if (!make_map(&mql, a.Qlo, a.nq, a.dim, BM) || !make_map(&mxl, a.Xlo, a.n_rows, a.dim, BN)) return cudaErrorInvalidValue;
    if (f16 ? (!make_map(&mqh, a.Q16, a.nq, a.dim, BM, true) || !make_map(&mxh, a.X16, a.n_rows, a.dim, BN, true))
            : (!make_map(&mqh, a.Qhi, a.nq, a.dim, BM) || !make_map(&mxh, a.Xhi, a.n_rows, a.dim, BN)))
        return cudaErrorInvalidValue;
    TcParams p{};
    p.f16 = f16 ? 1 : 0;
    static const bool no_cluster = getenv("PYROPE_FLAT_NOCLUSTER") != nullptr;
    const bool cluster = mode == 1 && !gmax && !no_cluster;
    static const int csize = getenv("PYROPE_FLAT_CLUSTER") ? atoi(getenv("PYROPE_FLAT_CLUSTER")) : 2;
    const int CS = csize == 4 ? 4 : 2;
    if (cluster && !make_map(&mxl, f16 ? a.X16 : static_cast<const void*>(a.Xhi), a.n_rows, a.dim, BN / CS, f16)) return cudaErrorInvalidValue;
    p.nq = a.nq; p.n_scan = a.n_scan; p.dim = a.dim; p.kprime = a.kprime; p.cap = a.cap; p.splits = splits;
    p.ntiles = (a.n_scan + BN - 1) / BN;
    p.tiles_per_split = (p.ntiles + splits - 1) / splits;
    p.gmax = gmax; p.gstride = p.ntiles * (BN / 32); p.tau_init = tau_init;
    p.halves = flat_tc_parts_per_split(a);
    p.one_term = ((gmax && a.amax) || mode == 1) ? 1 : 0;
    const int64_t nq_pad_f = flat_tc_nq_pad(a.nq);
    if (mode == 1) { p.band = a.tau_ws + nq_pad_f; p.overflow = reinterpret_cast<int*>(a.tau_ws + 2 * nq_pad_f); }
    if (mode == 2) p.run_if = reinterpret_cast<const int*>(a.tau_ws + 2 * nq_pad_f);
    p.has_uscale = (a.metric == kL2 || a.metric == kIP || !a.scale) ? 1 : 0;
    p.uscale = a.metric == kL2 && a.scale ? 2.f : 1.f;
    p.scale = a.scale; p.bias = a.bias; p.queue = a.queue; p.counts = a.counts;
    const int64_t qtiles = (a.nq + BM - 1) / BM;
    p.nq_pad = qtiles * BM;
    const size_t smem = (size_t)STAGES * STAGE_BYTES + 16 * 8 + 16 + 4 * (4 * BN * sizeof(float)) + 64;
    cudaError_t e = cudaFuncSetAttribute(flat_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (a.ev_k0 && !gmax && mode != 2) cudaEventRecord(a.ev_k0, st);
    if (cluster) {
        p.cluster = CS;
        p.qtiles_grid = (qtiles + CS - 1) / CS * CS;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)(p.qtiles_grid * splits));
        cfg.blockDim = dim3(TC_THREADS);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute at{};
        at.id = cudaLaunchAttributeClusterDimension;
        at.val.clusterDim.x = (unsigned)CS; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
        cfg.attrs = &at;
        cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, flat_tc_kernel, mqh, mql, mxh, mxl, p);
        if (e != cudaSuccess) return e;
    } else {
        flat_tc_kernel<<<(unsigned)(qtiles * splits), TC_THREADS, smem, st>>>(mqh, mql, mxh, mxl, p);
    }
    if (a.ev_k1 && !gmax && mode != 2) cudaEventRecord(a.ev_k1, st);
    return cudaGetLastError();
}

cudaError_t launch_flat_tc(const FlatTcParams& a, cudaStream_t st) {
    if (a.nq <= 0) return cudaSuccess;
    cudaError_t e = launch_flat_tc_select(a, st);
    if (e != cudaSuccess) return e;
    RescoreParams r{};
    r.Q = a.Q; r.nq = a.nq; r.dim = a.dim; r.X = a.X; r.xnorm = a.xnorm; r.qnorm = a.qnorm; r.labels = a.labels;
    r.metric = a.metric; r.k = a.k; r.cap = a.cap; r.splits = a.splits * flat_tc_parts_per_split(a); r.queue = a.queue; r.counts = a.counts;
    r.nq_pad = flat_tc_nq_pad(a.nq); r.out = a.out;
    // window of the re-score: room for the usual k' + band per query and at least 2k, never more than 4,096 keys
    // (32 KiB, so that many queries' CTAs stay resident); bigger totals take several rounds inside the kernel
    const int usual = a.kprime * 2 + 64;
    const int P = std::min(4096, next_pow2(std::max(std::max(2 * a.k, usual), 64)));
    r.arith = a.arith == 1 ? 1 : 2;
    flat_rescore_kernel<<<(unsigned)a.nq, 256, sizeof(uint64_t) * (size_t)P + sizeof(float) * (size_t)a.dim, st>>>(r, P);
    return cudaGetLastError();
}

}  // namespace pyrope
