// kernels.h — launchers of the sm_100a kernels behind libpyrope_gpu.so (internal; not the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pyrope {

enum Metric { kL2 = 0, kIP = 1, kCosine = 2 };

// Every scan kernel emits, per query and per "part" (a base split, a probe group, the buffer ...),
// its local top-k as (score, label) pairs into one combined array laid out [nq][parts_total][k];
// label < 0 marks an empty slot.  merge_pairs() then reduces parts_total*k -> k_out per query.
struct PairOut {
    float* scores;
    int64_t* labels;
    int parts_total;  // S
    int part_base;    // first part index this launch writes
};

// ---- K1: exact FLAT scan + top-k (CUDA-core path) -------------------------------------------
// Replaces BruteForceVectorIndex.Search:341-360 (and, over centroids, the coarse ranking at
// IvfFlatVectorIndex.cs:186-198 / IvfPqVectorIndex.cs:141-150).
struct FlatScanParams {
    const float* Q; int64_t nq; int dim;
    const float* X; int64_t n_scan;          // scan positions [0, n_scan)
    const uint8_t* dead;                     // nullable: non-zero = skip
    const float* xnorm; const float* qnorm;  // cosine only
    const int64_t* labels;                   // nullable: label = position
    int metric; int k;
    int splits;                              // parts written: [part_base, part_base+splits)
    uint64_t* queue; int cap;                // scratch [splits][nq][cap]
    PairOut out;
};
int flat_scan_cap(int k);
int flat_scan_pick_splits(int64_t nq, int64_t n_scan, int k, int num_sms, int max_parts);
cudaError_t launch_flat_scan(const FlatScanParams& p, cudaStream_t st);

// ---- K1 on tensor cores: 3xTF32 tcgen05 GEMM + fused top-k + exact fp32 re-score (flat_tc.cu) ----
struct FlatTcParams {
    const float* Q; const float* Qhi; const float* Qlo; int64_t nq; int dim;
    const float* X; const float* Xhi; const float* Xlo;
    int64_t n_rows;                          // rows backing X/Xhi/Xlo (tensor-map extent)
    int64_t n_scan;                          // scan positions [0, n_scan)
    const float* scale; const float* bias;   // per-row proxy terms (bias = -inf for tombstones)
    const float* xnorm; const float* qnorm;  // cosine re-score
    const int64_t* labels;
    int metric, k, kprime, cap, splits;
    int arith = 2;                           // re-score order: 1 = VectorMath.*Unsafe (FLAT index), 2 = L2Squared / DotProduct (IVF)
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;  // optional: recorded around the tcgen05 kernel alone
    uint64_t* queue; int32_t* counts;        // scratch [splits][nq_pad][cap], [splits][nq_pad]
    const float* amax = nullptr;             // optional: max_r |scale_r||x_r| of the operand => pass A runs 1xTF32
    // optional fp16 copies (launch_tc_half*) for the single one-term pass (L2 / IP, every table value within the fp16
    // range; qbad [nq] marks queries that are not): kind::f16 at twice the tf32 rate and half the operand bytes
    const void* Q16 = nullptr; const void* X16 = nullptr; const uint8_t* qbad = nullptr;
    float* gmax_ws = nullptr;                // optional two-pass threshold scratch: flat_tc_gmax_floats() floats
    float* tau_ws = nullptr;                 //   and flat_tc_nq_pad() floats (both set => two passes)
    PairOut out;                             // writes ONE part (splits are reduced by the re-score)
};
// two-pass threshold (group maxima -> per-query tau -> filtered pass): worth it only when the tile is
// epilogue-bound (small dim) and the stream is long
bool flat_tc_twopass(int dim, int64_t n_scan, int kprime);
// single one-TF32 pass with band pruning + exact re-score (tau_ws and amax set, gmax_ws null): long-K FLAT scans
bool flat_tc_oneterm(int dim, int64_t n_scan, int kprime);
size_t flat_tc_gmax_floats(int64_t nq, int64_t n_scan);
int flat_tc_pick_splits_seeded(int64_t nq, int64_t n_scan, int kprime, int num_sms);
bool flat_tc_supported(int dim, int k);
// queue / counts parts per (split, query): 2 on the two-pass path (column halves), else 1
int flat_tc_parts_per_split(const FlatTcParams& p);
int flat_tc_margin(int k);
int flat_tc_cap(int kprime);
int flat_tc_pick_splits(int64_t nq, int64_t n_scan, int kprime, int num_sms);
int64_t flat_tc_nq_pad(int64_t nq);
// hi = tf32(x) (round to nearest), lo = x - hi for rows [from_row, n); scale/bias may be null.  norms (cosine): the
// exact row norms [n] the re-score divides by; a row's proxy scale is 0 where they are below 1e-6
cudaError_t launch_tc_prepare(const float* X, int64_t n, int dim, int metric, const uint8_t* dead, float* hi,
                              float* lo, float* scale, float* bias, int64_t from_row, cudaStream_t st,
                              const float* norms = nullptr);
cudaError_t launch_tc_rowterms(const float* X, int64_t n, int dim, int metric, const uint8_t* dead, float* scale,
                               float* bias, cudaStream_t st, const float* norms = nullptr);
// amax (device float, zero-initialised) = max(amax, max over rows [from_row, n) of |scale_r| * |x_r|)
cudaError_t launch_tc_amax(const float* X, int64_t n, int dim, const float* scale, float* amax, int64_t from_row,
                           cudaStream_t st);
cudaError_t launch_flat_tc(const FlatTcParams& p, cudaStream_t st);
// selection only: leaves the k' best proxy candidates per (split, query) sorted in queue/counts
cudaError_t launch_flat_tc_select(const FlatTcParams& p, cudaStream_t st);
// bit-exact arg-best among the shortlisted centroids of each row (split 0 of queue/counts), in the
// reference's evaluation order; flag[row] = 1 when the shortlist may be incomplete (full and its
// last proxy score within eps of the first) so the caller re-runs that row exhaustively.
cudaError_t launch_assign_from_shortlist(int metric, int dim, int64_t n, const float* X, int64_t ldx,
                                         const float* centroids, const float* cnorms, const uint64_t* queue,
                                         const int32_t* counts, int cap, int kprime, int32_t* assign,
                                         uint8_t* flag, cudaStream_t st);
// scatter: dst[idx[i]] = src[i]
cudaError_t launch_scatter_i32(const int32_t* src, const int64_t* idx, int64_t n, int32_t* dst, cudaStream_t st);

// ---- coarse probe of a batched IVF search, query tile resident in shared memory (coarse_tc.cu) -----------------
// Replaces the centroid ranking of IvfFlatVectorIndex.cs:186-198 / IvfPqVectorIndex.cs:141-150 for a batch: one-TF32
// tensor-core scores pick the few centroids per query that can be among the nprobe best, those are ranked in the
// reference's own arithmetic.  probes_out [nq][nprobe] list ids, best first, -1 = none.
constexpr int kCoarseTcCap = 512;     // candidate positions kept per query before the exhaustive fallback
constexpr int kCoarseTcMargin = 8;    // k' = nprobe + margin unit maxima bound the threshold
struct CoarseTcParams {
    const float* Q; const float* Qhi; int64_t nq; int dim; int metric;
    const float* C; const float* Chi; const float* cnorms; int64_t nc;
    const float* scale; const float* bias; const float* amax;   // proxy terms of the centroid operand (TcOperand)
    // optional fp16 copies of both operands (launch_tc_half*): the tensor passes then run kind::f16.  Only for tables whose
    // values all fit the fp16 range; qbad [nq] marks queries that do not (they are ranked exhaustively).  L2 / IP only.
    const void* Q16 = nullptr; const void* C16 = nullptr; const uint8_t* qbad = nullptr;
    int nprobe; int64_t* probes_out;
    void* scratch; int num_sms;
};
bool coarse_tc_supported(int dim, int64_t nc, int nprobe);
// fp16 copy of a table, round to nearest, saturating; absmax (device, zero-initialised by the caller) receives max |x|
cudaError_t launch_tc_half(const float* X, int64_t n_elems, void* out16, float* absmax, cudaStream_t st);
// the same per query row; bad[q] = 1 when a component of row q lies beyond the range the fp16 passes are proven for
cudaError_t launch_tc_half_rows(const float* Q, int64_t nq, int dim, void* out16, uint8_t* bad, cudaStream_t st);
constexpr float kTcHalfMaxAbs = 32768.f;
size_t coarse_tc_scratch_bytes(int64_t nq, int64_t nc, int num_sms);
int coarse_tc_launches();
cudaError_t launch_coarse_tc(const CoarseTcParams& p, cudaStream_t st);

// ---- FLAT, 8-bit scalar quantised (sq8.cu): ScalarQuantizer.Quantize:22-62 and the quantised branch of
// BruteForceVectorIndex.Search:297-336 (integer distances between byte vectors, VectorMath.cs:441-680)
cudaError_t launch_sq8_quantize(const float* X, int64_t n, int dim, int64_t ldx, uint8_t* out, int dpad, uint8_t* qvalid,
                                cudaStream_t st);
int sq8_pick_splits(int64_t nq, int64_t n_scan, int k, int num_sms);
cudaError_t launch_sq8_scan(const uint8_t* Q8, int64_t nq, int dpad, const uint8_t* X8, int64_t n_scan, const uint8_t* dead,
                            const uint8_t* qvalid, const int64_t* labels, int metric, int k, int splits, PairOut out,
                            cudaStream_t st);

// ---- K6: merge ------------------------------------------------------------------------------
// in: candidate (score,label) at address part*part_stride + q*q_stride + j, j < k_in.
// dedupe: a candidate whose label already occurs in a LOWER part is dropped (DeltaVectorIndex.cs:98-110: the
// head's copy of an id replaces the tail's).
// k_per_query (nullable, device [nq]): query q sees only entries j < k_per_query[q] of each part and keeps at most that
// many, so counts[q] <= k_per_query[q] — the merge a batch whose callers asked for different topK needs.
cudaError_t launch_merge_pairs(int64_t nq, int parts, int k_in, int k_out, const float* in_scores,
                               const int64_t* in_labels, int64_t part_stride, int64_t q_stride,
                               float* out_scores, int64_t* out_labels, int32_t* out_counts,
                               cudaStream_t st, bool dedupe = false, const int32_t* k_per_query = nullptr);
constexpr int kMergeMaxCandidates = 4096;

// ---- K4: IVF_FLAT inverted-list scan ----------------------------------------------------------
// Replaces IvfFlatVectorIndex.Search:200-218.
struct IvfFlatScanParams {
    const float* Q; int64_t nq; int dim;
    const int64_t* probes; int nprobe;       // [nq][nprobe] list ids in rank order, <0 = none
    const int32_t* allow;                    // nullable [nq][nprobe]: entries allowed per probe (MaxScans)
    const int64_t* list_off;                 // [nlist+1]
    const float* vecs; const uint8_t* dead; const float* norms; const int64_t* labels;
    const float* qnorm;
    int metric; int k; int groups;           // grid.y: probe groups (parts)
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;  // optional: recorded around the list-major scan kernel alone
    PairOut out;
};
cudaError_t launch_ivfflat_scan(const IvfFlatScanParams& p, cudaStream_t st);
// List-major variant (ivf_lm.cu): pairs grouped by list, 16 queries share one pass over a list's rows; writes
// ONE part.  L2 / inner product, dim % 4 == 0 and dim <= 128, no MaxScans budget.
bool ivfflat_lm_supported(int dim, int metric, int nprobe, int k, int64_t nq, int64_t list_total, bool has_budget);
size_t ivfflat_lm_scratch_bytes(int64_t nq, int nprobe, int k, int nlist);
int ivfflat_lm_launches();
cudaError_t launch_ivfflat_scan_lm(const IvfFlatScanParams& p, int nlist, void* scratch, int num_sms, cudaStream_t st);
cudaError_t ivfflat_lm_scanned_rows(const void* scratch, int64_t nq, int nprobe, int k, int nlist, unsigned long long* out,
                                    cudaStream_t st);

// ---- K5: IVF_PQ LUT build + ADC scan ----------------------------------------------------------
// Replaces ProductQuantizer.ComputeDistanceTable:98-120 + IvfPqVectorIndex.Search:152-199.
struct IvfPqScanParams {
    const float* Q; int64_t nq; int dim;
    const int64_t* probes; int nprobe;
    const int64_t* list_off; int nlist;
    int64_t max_list_len;                    // longest inverted list (list-major path sizing)
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;  // optional: recorded around the list-major scan kernel alone
    cudaStream_t aux_stream = nullptr;             // optional side stream (+ fork/join events): the threshold seed
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;  // kernel overlaps the grouping / item-block kernels
    const float* centroids;                  // [nlist][dim]
    const float* codebook; int m; int ksub;  // [m][ksub][dim/m]
    const float* cmax = nullptr;             // optional [16]: max codeword norm per sub-quantiser (launch_pq_cmax), cached per index
    // list-major path, m < 16 (m divides 16): the scan runs on the EQUIVALENT 16-table quantiser - every codeword cut
    // into 16/m pieces of dim/16 dimensions, every code byte repeated 16/m times (launch_pq_lm_expand_*): the same
    // squared distance, summed in 16 parts instead of m.  Only the approximate stages read these two; the final
    // re-score uses `codebook` / `codes` in the reference's own order.  nullptr when m = 16.
    const float* lm_codebook = nullptr;      // [16][ksub][dim/16]
    const uint8_t* lm_codes = nullptr;       // [total][16]
    const uint8_t* codes; const uint8_t* dead; const int64_t* labels;
    int k; int groups;
    int force_generic;                       // tests: run the simple kernel
    PairOut out;
    int32_t* out_counts = nullptr;           // list-major path only: results per query, when `out` is the final output
    // list-major path, multi-GPU: thresholds shared between the ranks WHILE the scan kernels run.  A bound one rank
    // proves for query q (k candidates at or below it) holds on every rank, so each tightening is also written,
    // with atomicMax over NVLink peer memory, into the peers' published arrays; thr_pub is this rank's own array
    // (what the peers write into), read next to the local threshold.  All nullptr / 0 on one GPU.
    // Words are (batch epoch << 32 | ordered bound), written with a 64-bit atomicMax: only words of the reader's own
    // batch count, so no clearing and no ordering between batches is needed for correctness.
    unsigned long long* thr_pub = nullptr;
    unsigned long long* peer_thr[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int n_peers = 0;
    uint32_t epoch = 0;
};
cudaError_t launch_ivfpq_scan(const IvfPqScanParams& p, cudaStream_t st);
// List-major variant (pq_lm.cu): (query, probe) pairs grouped by list, four queries per work item share
// one pass over the list's codes; writes ONE part (p.groups is ignored).  m in {1, 2, 4, 8, 16}, dim/16 in {4, 8}.
bool ivfpq_lm_supported(int dim, int m, int ksub, int nprobe, int k, int64_t nq, int64_t list_total, int64_t max_list_len);
size_t ivfpq_lm_scratch_bytes(int64_t nq, int nprobe, int k, int nlist, int dim, int64_t max_list_len);
int ivfpq_lm_launches();
cudaError_t launch_pq_lm_expand_codebook(const float* codebook, int m, int ksub, int dim, float* cb16, cudaStream_t st);
cudaError_t launch_pq_lm_expand_codes(const uint8_t* codes, int64_t n, int m, uint8_t* codes16, cudaStream_t st);
cudaError_t ivfpq_lm_scanned_codes(const void* scratch, int64_t nq, int nprobe, int k, int nlist, int dim,
                                   int64_t max_list_len, unsigned long long* out, cudaStream_t st);
cudaError_t launch_ivfpq_scan_lm(const IvfPqScanParams& p, void* scratch, int num_sms, cudaStream_t st);
// max_e |codeword(m, e)| for the 16 sub-quantisers of the list-major path (depends on the codebook only)
cudaError_t launch_pq_cmax(const float* codebook, int ksub, int sub, float* cmax16, cudaStream_t st);
// ProductQuantizer.ComputeDistanceTable for nq queries (parity tests): table [nq][m][k]
cudaError_t launch_pq_distance_table(const float* Q, int64_t nq, int dim, const float* codebook,
                                     int m, int k, float* table, cudaStream_t st);

// ---- MaxScans bookkeeping (IvfFlatVectorIndex.cs:172,202,209) ---------------------------------
cudaError_t launch_probe_allow(const int64_t* probes, int64_t nq, int nprobe,
                               const int64_t* list_off, int64_t budget, int32_t* allow,
                               cudaStream_t st);

// ---- bit-exact build kernels -------------------------------------------------------------------
// KMeansUtils.FindNearestCentroid:70-93 (VectorMath.L2Squared/DotProduct/Cosine order, no FMA)
cudaError_t launch_assign_exact(int metric, int dim, int64_t n, const float* X, int64_t ldx,
                                int nc, const float* centroids, const float* cnorms,
                                int32_t* assign, cudaStream_t st);
// exact-order re-ranking of the coarse stage's candidate lists (P_in >= P_out), best first, ties to the lower index;
// scores_in (stage-one scores, sorted descending) lets queries whose probed set is already settled skip it
// unless need_order is set
cudaError_t launch_coarse_rerank_exact(int metric, int dim, int64_t nq, const float* Q, const float* centroids,
                                       const float* cnorms, const int64_t* probes_in, const float* scores_in, int P_in,
                                       int64_t* probes_out, float* scores_out, int P_out, int need_order, cudaStream_t st);
// ComputeNorm:72-100 in the reference's order, one row per thread group
cudaError_t launch_row_norms_exact(const float* X, int64_t n, int dim, int64_t ldx, float* out,
                                   cudaStream_t st);
// residual = x - centroid[assign]   (IvfPqVectorIndex.cs:82-85)
cudaError_t launch_residuals(const float* X, int64_t n, int dim, const float* centroids,
                             const int32_t* assign, float* out, cudaStream_t st);
// ProductQuantizer.Encode:60-80 + FindNearest:122-136 (L2SquaredUnsafe order, no FMA)
cudaError_t launch_pq_encode_exact(const float* R, int64_t n, int dim, int m, int kpad,
                                   const float* codebook, const int32_t* ksub, uint8_t* codes,
                                   cudaStream_t st);
// KMeansUtils.Train:46-63 update: order[offs[c]..offs[c+1]) lists the rows of cluster c in data
// order; fp32 running sums in that order, /= count, ArraysEqual(1e-6) gate.  changed: int flag.
cudaError_t launch_kmeans_update(const float* X, int64_t ldx, int dim, int nc,
                                 const int64_t* offs, const int32_t* order, float* centroids,
                                 int* changed, cudaStream_t st);
// gather rows: out[i] = X[idx[i]]  (rows of `width` elements of `elem` bytes)
cudaError_t launch_gather_rows(const void* X, int64_t row_bytes, const int64_t* idx, int64_t n,
                               void* out, cudaStream_t st);
// scatter rows: out[idx[i]] = X[i]
cudaError_t launch_scatter_rows(const void* X, int64_t row_bytes, const int64_t* idx, int64_t n,
                                void* out, cudaStream_t st);
// where[i] = index of labels[i] in the ascending array sorted[ns], or -1 (also -1 where skip[i] != 0)
cudaError_t launch_find_labels(const int64_t* labels, const uint8_t* skip, int64_t n, const int64_t* sorted,
                               int64_t ns, int64_t* where, cudaStream_t st);
cudaError_t launch_iota64(int64_t* out, int64_t n, int64_t base, cudaStream_t st);

// ---- Extend: list merge (extend.cu) -----------------------------------------------------------
// One column = one list-major array (payload, row ordinals, labels, dead flags, norms) of row_bytes per entry.  Merged
// list c starts at off_merged[c] = off_old[c] + offs_new[c]: old entry i of list c moves to i + offs_new[c], new sorted
// entry j (0-based within list c) goes to off_old[c + 1] + j, taken from row order[offs_new[c] + j] of new_src (buffer
// order, [n][row_bytes]; nullptr writes zeros).  fold_flags: every non-zero old byte becomes 1 (shadowed -> deleted).
constexpr int kExtendMaxColumns = 5;
struct ExtendMergeColumn {
    const uint8_t* old_src; const uint8_t* new_src; uint8_t* dst;
    int64_t row_bytes; int fold_flags;
    int64_t tile0;                           // set by the launcher
};
struct ExtendMergeParams {
    const int64_t* off_old; const int64_t* offs_new; const int64_t* off_merged;  // [nc + 1] each
    const int32_t* order; int nc; int ncols;
    ExtendMergeColumn col[kExtendMaxColumns];
};
// CTAs of the merge for one column (16 KiB of merged bytes each)
int64_t extend_merge_tiles(int64_t merged_rows, int64_t row_bytes);
cudaError_t launch_extend_merge(ExtendMergeParams p, int64_t merged_rows, cudaStream_t st);
cudaError_t launch_fill_uniform(float* out, int64_t n, uint64_t seed, uint64_t offset,
                                cudaStream_t st);

}  // namespace pyrope
