/*
 * pyrope_gpu.h — C ABI of libpyrope_gpu.so: B200 (sm_100a) implementation of Pyrope's vector-scan
 * hot path (FLAT exact scan, IVF_FLAT coarse-assign + inverted-list scan, IVF_PQ ADC scan, each with
 * top-k), behind the reference's IVectorIndex surface.
 *
 * The reference (takurot/Pyrope) is 100 % managed C# and has NO FFI today; the seam this ABI plugs
 * into is the interface src/Pyrope.GarnetServer/Vector/IVectorIndex.cs:14-29 (+ ICentroidsProvider.cs:9-15),
 * constructed in exactly one place, Services/VectorIndexRegistry.cs:81-113.  A C# class
 * Gpu*VectorIndex : IVectorIndex P/Invokes the functions below (stub in INTEGRATION.md).
 *
 * Conventions
 *  - every function returns a pyrope_status (0 ok, <0 error); pyrope_last_error() returns a
 *    thread-local message.  The library never aborts/exits (VectorCommandSet.cs:547-554 turns any
 *    exception into "-ERR <message>"; the shim maps codes to the .NET exception types named below).
 *  - host pointers unless the function name ends in _device.  Inputs are only read during the call
 *    (the library copies, as BruteForceVectorIndex.Add does, BruteForceVectorIndex.cs:147-148).
 *  - string ids stay host-side in the shim (List<string>/Dictionary<string,long> exactly like
 *    BruteForceVectorIndex.cs:14-15); the library deals in dense int64 ROW ordinals that it assigns
 *    at add time (0,1,2,... per index), plus an optional caller-chosen int64 LABEL per row that
 *    search returns instead of the ordinal (used for global row numbers when sharded across GPUs).
 *  - scores are "higher is better" for every metric: L2 -> -||q-x||^2, InnerProduct -> q.x,
 *    Cosine -> q.x/(|q||x|) (0 if either norm < 1e-6), as in the reference.
 *  - a pyrope_index lives on one GPU.  N GPUs: one process drives them all through pyrope_sharded_*,
 *    or one process per GPU shards with pyrope_index_set_shard and exchanges probe lists / top-k lists
 *    with pyrope_peer_* (peer stores over NVLink) or any all-gather of its own.  Search is thread-safe
 *    for concurrent callers on one handle, mutation must be serialised by the caller (the shim's
 *    ReaderWriterLockSlim already does).
 */
#ifndef PYROPE_GPU_H
#define PYROPE_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pyrope_index pyrope_index; /* opaque */
typedef struct pyrope_sharded pyrope_sharded;     /* one index over the GPUs of a box, below */
typedef struct pyrope_delta pyrope_delta;         /* Head+Tail, below */
typedef struct pyrope_vindex pyrope_vindex;       /* string-id index classes, below */

typedef enum pyrope_status {
    PYROPE_OK = 0,
    PYROPE_ERR_INVALID_ARG = -1,   /* -> ArgumentException / ArgumentNullException            */
    PYROPE_ERR_DIMENSION = -2,     /* -> ArgumentException("Vector dimension mismatch") => VEC_ERR_DIM */
    PYROPE_ERR_OUT_OF_RANGE = -3,  /* -> ArgumentOutOfRangeException (topK <= 0, dim <= 0)     */
    PYROPE_ERR_INVALID_STATE = -4, /* -> InvalidOperationException (e.g. "PQ not trained")     */
    PYROPE_ERR_NOT_FOUND = -5,     /* row does not exist / already deleted                    */
    PYROPE_ERR_CUDA = -6,          /* CUDA runtime failure; message carries cudaGetErrorString */
    PYROPE_ERR_OOM = -7,           /* device or host allocation failed                         */
    PYROPE_ERR_UNSUPPORTED = -8    /* shape outside what the kernels cover (documented limits) */
} pyrope_status;

/* VectorIndexRegistry.cs:87-108 picks the tail by Algorithm string; these are the GPU kinds. */
typedef enum pyrope_kind { PYROPE_FLAT = 0, PYROPE_IVF_FLAT = 1, PYROPE_IVF_PQ = 2 } pyrope_kind;
/* IVectorIndex.cs:5-10 VectorMetric (same numeric values) */
typedef enum pyrope_metric { PYROPE_L2 = 0, PYROPE_INNER_PRODUCT = 1, PYROPE_COSINE = 2 } pyrope_metric;

/* ---- process / device ------------------------------------------------------------------- */
/* Select the CUDA device this process drives and warm the context.  device < 0 keeps the current. */
int pyrope_gpu_init(int device);
int pyrope_gpu_shutdown(void);
int pyrope_gpu_device_count(int *out);
const char *pyrope_last_error(void);
int pyrope_version(void);

/* ---- lifecycle: replaces the index constructors (BruteForceVectorIndex.cs:42-51,
 *      IvfFlatVectorIndex.cs:27-33 nList=100, IvfPqVectorIndex.cs:27-35; registry defaults
 *      m=4,k=256,nlist=100 at VectorIndexRegistry.cs:96-106).  nlist/pq_m/pq_k ignored for FLAT. */
int pyrope_index_create(int kind, int dim, int metric, int nlist, int pq_m, int pq_k,
                        pyrope_index **out);
int pyrope_index_destroy(pyrope_index *h);
/* Pre-size device storage for n_rows raw vectors (optional; avoids regrowth copies). */
int pyrope_index_reserve(pyrope_index *h, int64_t n_rows);

/* ---- writes: replace IVectorIndex.Add / Upsert / Delete ----------------------------------- */
/* Append n vectors (X is n x dim row-major).  labels may be NULL (label = row ordinal).
 * FLAT: rows join the scan order at the end (BruteForceVectorIndex.cs:162-184 InternalAdd).
 * IVF_*: rows join the pre-build buffer (IvfFlatVectorIndex.cs:39-55, IvfPqVectorIndex.cs:36-45),
 *        re-using freed buffer slots LIFO like Dictionary<,> does so enumeration order matches.
 * first_row_out receives the ordinal of the first appended row (ordinals are consecutive). */
int pyrope_index_add_batch(pyrope_index *h, int64_t n, const float *X, const int64_t *labels,
                           int64_t *first_row_out);
int pyrope_index_add_batch_device(pyrope_index *h, int64_t n, const float *dX,
                                  const int64_t *d_labels, int64_t *first_row_out);
/* Overwrite a live (or, for FLAT, tombstoned: Upsert un-deletes, BruteForceVectorIndex.cs:200-203)
 * row in place: Upsert of an existing id keeps its scan position.  IVF rows must be in the buffer. */
int pyrope_index_update_row(pyrope_index *h, int64_t row, const float *x);
/* Tombstone a row (BruteForceVectorIndex.cs:231-254; IvfFlatVectorIndex.cs:62-83).
 * IVF_PQ mirrors the reference: only buffer rows can be deleted (IvfPqVectorIndex.cs:48-53);
 * a row already encoded into a list returns PYROPE_ERR_NOT_FOUND. */
int pyrope_index_delete_row(pyrope_index *h, int64_t row);
/* Hide (1) / unhide (0) a list row that a newer buffer row with the same id shadows
 * (the seenIds skip at IvfFlatVectorIndex.cs:210, IvfPqVectorIndex.cs:170). */
int pyrope_index_shadow_row(pyrope_index *h, int64_t row, int shadowed);

/* Replace the label of every row: labels_by_row[r] for row ordinal r, n_rows >= rows ever added.  Used after
 * pyrope_index_load by a shim whose labels are process-local id ordinals. */
int pyrope_index_set_labels(pyrope_index *h, int64_t n_rows, const int64_t *labels_by_row);

/* BruteForceVectorIndex.EnableQuantization (BruteForceVectorIndex.cs:23-40), FLAT only: while on, added / upserted
 * rows also get an 8-bit copy (ScalarQuantizer.Quantize, ScalarQuantizer.cs:22-62: per-vector min / max) and Search
 * ranks by the integer distance between the quantised query and the quantised rows (:297-336: -L2Squared8Bit for
 * L2, DotProduct8Bit for inner product and cosine).  Rows written while it was off have no quantised form: MaxScans
 * counts them, results never contain them (:312-322). */
int pyrope_index_set_quantization(pyrope_index *h, int enable);

/* ---- build: replaces IVectorIndex.Build (IvfFlatVectorIndex.cs:85-145, IvfPqVectorIndex.cs:55-116;
 *      FLAT is a no-op, BruteForceVectorIndex.cs:56).  Training follows KMeansUtils.Train
 *      (KMeansUtils.cs:10-68: System.Random init seed 42 / 123 / 42+m, <=10 Lloyd iterations,
 *      fp32 means in data order) and ProductQuantizer.Train/Encode (ProductQuantizer.cs:28-80)
 *      bit-exactly on device unless codebooks were frozen with pyrope_index_set_codebooks. */
int pyrope_index_build(pyrope_index *h);
/* Bound the training set to the first max_train_rows rows (<=0: all, the reference rule) and the
 * Lloyd iterations (<=0: 10, the reference default).  Opt-in deviation for very large builds. */
int pyrope_index_set_train_params(pyrope_index *h, int64_t max_train_rows, int max_iter);
/* Extend (opt-in, no counterpart in the reference): append the write buffer to the inverted lists of a BUILT IVF index
 * without re-training — FAISS's "add to a trained index".  Every live buffer row, in slot order, goes to its nearest
 * CURRENT centroid (the bit-exact assignment Build uses); IVF_PQ rows are encoded with the CURRENT codebooks (ksub
 * honoured).  Each row is appended to the END of its list, rows of one list in slot order, and keeps its row ordinal.
 * Existing entries keep their positions, row ordinals, labels and dead flags (nothing is compacted, so MaxScans walks
 * old entries in the same order), except that shadowed entries become deleted: their replacements have just left the
 * buffer.  The buffer is emptied; centroids, codebooks and next row ordinal are unchanged.  A shard
 * (pyrope_index_set_shard) appends only to the lists it owns and empties its replica of the buffer.  All or nothing:
 * on any error the index is exactly as it was.  FLAT -> UNSUPPORTED, not built -> INVALID_STATE, empty buffer -> OK. */
int pyrope_index_extend(pyrope_index *h);
/* Freeze codebooks as given inputs: centroids [n_centroids][dim]; pq_codebooks [m][k][dim/m]
 * (NULL for IVF_FLAT).  The next pyrope_index_build only assigns (+ encodes). */
int pyrope_index_set_codebooks(pyrope_index *h, int n_centroids, const float *centroids,
                               const float *pq_codebooks);
/* Multi-GPU sharding of an IVF index (SURVEY §8e): this process keeps only the inverted lists with
 * list_id % world == rank (centroids and PQ codebooks stay replicated); rows assigned to other lists
 * are dropped at the next pyrope_index_build.  Every rank sees all rows and all queries; per-rank
 * top-k lists are all-gathered (pyrope_peer_allgather_device, or NCCL) and reduced by pyrope_topk_merge_device. */
int pyrope_index_set_shard(pyrope_index *h, int rank, int world);
/* Multi-GPU IVF_PQ (list-major scan): share per-query thresholds between the ranks while their scan kernels run.  A
 * bound one rank proves for a query (k candidates at or below it) holds on every rank, so every tightening is also
 * written with a 64-bit atomicMax into the peers' published arrays over NVLink peer memory — the one exchange on this
 * path that lives inside a kernel.  Each rank: _handle (allocates its array for batches of up to max_queries queries,
 * returns a 64-byte CUDA IPC handle), all-gather the handles, _open (handles = world x 64 bytes, own slot ignored).
 * PRECONDITION: every rank searches the SAME sequence of batches with pyrope_index_search_batch_probed_device.  Each
 * published word is (batch epoch << 32 | bound) and a rank only believes words of the epoch it is searching, so ranks
 * need NOT be ordered against each other between batches: a peer that is still in an earlier batch (or already in a
 * later one) cannot prune this one.  The epoch is a per-handle counter of probed searches made while peers are attached
 * (starts at 1); a caller whose ranks might not count alike names it itself with _epoch (non-zero, increasing) before
 * each search.  A shard may return fewer than k rows (the rest cannot be in the global top k). */
int pyrope_index_threshold_exchange_handle(pyrope_index *h, int64_t max_queries, void *handle_out);
int pyrope_index_threshold_exchange_open(pyrope_index *h, int world, int rank, const void *handles);
int pyrope_index_threshold_exchange_close(pyrope_index *h); /* stop publishing / reading; the own array stays mapped */
int pyrope_index_threshold_exchange_epoch(pyrope_index *h, uint32_t epoch); /* epoch of the NEXT probed search */
/* The same exchange between indexes of ONE process (pyrope_sharded_*): _array (re)allocates this index's array and returns
 * its device pointer, _attach takes every shard's pointer (world entries, own slot ignored; peer access between the
 * devices must be enabled).  _close detaches. */
int pyrope_index_threshold_exchange_array(pyrope_index *h, int64_t max_queries, void **d_array_out);
int pyrope_index_threshold_exchange_attach(pyrope_index *h, int world, int rank, void *const *arrays);
int pyrope_index_is_built(pyrope_index *h, int *out);
/* ICentroidsProvider.GetCentroids (IvfFlatVectorIndex.cs:314-325): n_out = 0 until built.
 * centroids_out may be NULL to query the count. */
int pyrope_index_get_centroids(pyrope_index *h, float *centroids_out, int *n_out);
/* pq codebooks [m][k][dim/m] (zero padded) and trained codewords per subspace ksub[m]. */
int pyrope_index_get_codebooks(pyrope_index *h, float *codebooks_out, int32_t *ksub_out);
/* Inverted-list layout for parity checks: offsets [n_centroids+1]; rows (ordinals) and, for IVF_PQ,
 * codes [total][m], both list-major in list order.  Any output may be NULL. total_out = entries. */
int pyrope_index_get_lists(pyrope_index *h, int64_t *offsets_out, int64_t *rows_out,
                           uint8_t *codes_out, int64_t *total_out);

/* ---- snapshot / load: replace IVectorIndex.Snapshot / Load (BruteForceVectorIndex.cs:58-107,
 *      IvfFlatVectorIndex.cs:233-298; IVF_PQ's are no-ops in the reference, IvfPqVectorIndex.cs:228-229).
 *      One binary file per index, written to path + ".tmp" and moved into place like DeltaVectorIndex.cs:160-212
 *      does.  load() requires an index created with the same kind / dim / metric / m / k and replaces its whole
 *      state (rows, tombstones, trained codebooks, inverted lists).  Missing file -> NOT_FOUND
 *      (FileNotFoundException in the shim), foreign file -> INVALID_ARG. */
int pyrope_index_snapshot(pyrope_index *h, const char *path);
int pyrope_index_load(pyrope_index *h, const char *path);

/* ---- stats: replaces IVectorIndex.GetStats (O(1), host-side, never a device sync;
 *      BruteForceVectorIndex.cs:119-131, IvfFlatVectorIndex.cs:300-312).  live_rows counts every
 *      searchable row; the shim reproduces IvfPqVectorIndex.cs:230's hard-coded 0 itself. */
int pyrope_index_stats(pyrope_index *h, int64_t *live_rows, int64_t *buffer_rows, int *dim,
                       int *metric);

/* ---- search: replaces IVectorIndex.Search for nq queries at once (VectorCommandSet.cs:458 calls it
 *      one query at a time; the host micro-batcher funnels concurrent callers into this).
 *      Q is nq x dim.  max_scans < 0 = SearchOptions.MaxScans null; nprobe < 0 = NProbe null
 *      (defaults 3 / 1: IvfFlatVectorIndex.cs:14, IvfPqVectorIndex.cs:125).
 *      Outputs are nq x topk, best first; slots past counts[i] hold score 0 / row -1.
 *      Errors: topk <= 0 -> OUT_OF_RANGE for FLAT (BruteForceVectorIndex.cs:278), empty result for
 *      IVF (no validation in the reference); topk > 1024 -> UNSUPPORTED. */
int pyrope_index_search_batch(pyrope_index *h, int64_t nq, const float *Q, int topk,
                              int64_t max_scans, int nprobe, float *scores_out, int64_t *rows_out,
                              int32_t *counts_out);
/* Same with device-resident queries/outputs, enqueued on `stream` (a cudaStream_t; NULL = the
 * library's own stream, synchronised before return). */
int pyrope_index_search_batch_device(pyrope_index *h, int64_t nq, const float *dQ, int topk,
                                     int64_t max_scans, int nprobe, float *d_scores,
                                     int64_t *d_rows, int32_t *d_counts, void *stream);
/* Multi-GPU split of a batched IVF search (SURVEY §8e): the coarse ranking of IvfFlatVectorIndex.cs:186-198 /
 * IvfPqVectorIndex.cs:141-150 depends only on the replicated centroids, so each rank ranks centroids for
 * ITS slice of the batch (coarse_probe), the probe lists are all-gathered (nq x nprobe int64, list ids in
 * rank order, -1 = none; nprobe must be the effective value, >= 1), and every rank scans its list shard
 * for ALL queries with the gathered probes (search_batch_probed).  Device pointers. */
int pyrope_index_coarse_probe_device(pyrope_index *h, int64_t nq, const float *dQ, int nprobe,
                                     int64_t *d_probes_out, void *stream);
int pyrope_index_search_batch_probed_device(pyrope_index *h, int64_t nq, const float *dQ, int topk,
                                            int64_t max_scans, int nprobe, const int64_t *d_probes,
                                            float *d_scores, int64_t *d_rows, int32_t *d_counts,
                                            void *stream);
/* Kernel-only time (ms, CUDA events) of the most recent search on this handle, split by stage:
 * out[0]=total, [1]=coarse probe, [2]=list/base scan, [3]=merge.  Feeds TraceInfo (SURVEY §5). */
int pyrope_index_last_search_ms(pyrope_index *h, float *out4);
/* CUDA-event duration (ms) of the DOMINANT kernel of the most recent search alone (the list-major
 * ADC scan kernel for IVF_PQ, the tcgen05 kernel for FLAT) and its name ("" / 0 if the search took
 * another path).  Measurement only: feeds the bench's roofline figure. */
int pyrope_index_last_search_kernel(pyrope_index *h, float *ms_out, const char **name_out);
/* Number of kernel launches issued by the most recent search on this handle. */
int pyrope_index_last_search_launches(pyrope_index *h, int *out);
/* PQ codes scored by the most recent batched IVF_PQ search (sum over its (query, probe) pairs of the
 * probed list's length; 0 if the search did not take the list-major path).  Measurement only: this is
 * the unit count behind the bench's algorithmic HBM bytes (m bytes per scored code). */
int pyrope_index_last_search_scanned(pyrope_index *h, int64_t *codes_out);

/* ---- host micro-batcher: the reference calls IVectorIndex.Search with ONE query per Garnet session thread
 *      (VectorCommandSet.cs:458, under the read lock of BruteForceVectorIndex.cs:282).  The shim's Search calls
 *      pyrope_batcher_search instead, which blocks while a dispatcher thread gathers the queries that arrive
 *      within max_wait_us (or max_batch of them), issues one batched search of its target per group of equal
 *      (MaxScans, NProbe, K) and returns each caller its own result.  K is the topK class: the smallest power of two
 *      >= topK, capped at the target's limit; a group is searched once at its largest topK and every caller gets
 *      exactly its own top topK (a Head+Tail merges with a per-query k, pyrope_delta_search_batch_topk).
 *      Thread-safe; results are written into the caller's buffers (topk entries each); errors carry
 *      pyrope_batcher_last_error(), with the message of whichever layer raised them.
 *      The target is borrowed: destroy the batcher first.  It is one of
 *        pyrope_batcher_create          a pyrope_index: rows_out = row ordinals (or the rows' labels);
 *        pyrope_batcher_create_sharded  a pyrope_sharded: global row ordinals (labels), dimension from shard 0;
 *        pyrope_batcher_create_delta    a pyrope_delta (Head+Tail): labels, dimension from the head;
 *        pyrope_batcher_create_vindex   a pyrope_vindex (string ids): id ORDINALS.  The batch runs under the vindex's
 *                                       shared lock, as pyrope_vindex_search does.  The shim checks the query length
 *                                       itself (ValidateDim) before it calls pyrope_batcher_search, holds its read lock
 *                                       while blocked in it, and turns the ordinals into strings with pyrope_vindex_ids
 *                                       before it releases that lock.
 *      A caller's status is the one the direct call on the target would give it alone, and such callers never join a
 *      batch: topK <= 0 -> OUT_OF_RANGE on a FLAT index, a delta, or a vindex whose search validates like a FLAT head,
 *      an empty result on an IVF index or leaf; topK above the target's limit (1024 for an index, min(1024, 4096 / N)
 *      sharded, what pyrope_delta_search_batch accepts for a delta) -> UNSUPPORTED.  A batch that fails reports its
 *      status and message to every caller in it.  A null target -> INVALID_ARG before any CUDA call. */
typedef struct pyrope_batcher pyrope_batcher;
int pyrope_batcher_create(pyrope_index *h, int max_batch, int max_wait_us, pyrope_batcher **out);
int pyrope_batcher_create_sharded(pyrope_sharded *s, int max_batch, int max_wait_us, pyrope_batcher **out);
int pyrope_batcher_create_delta(pyrope_delta *d, int max_batch, int max_wait_us, pyrope_batcher **out);
int pyrope_batcher_create_vindex(pyrope_vindex *v, int max_batch, int max_wait_us, pyrope_batcher **out);
int pyrope_batcher_destroy(pyrope_batcher *b);
int pyrope_batcher_search(pyrope_batcher *b, const float *query, int topk, int64_t max_scans, int nprobe,
                          float *scores_out, int64_t *rows_out, int32_t *count_out);
int pyrope_batcher_stats(pyrope_batcher *b, int64_t *batches_out, int64_t *queries_out);
const char *pyrope_batcher_last_error(void);

/* ---- cross-shard merge (the step after the all-gather of the per-shard lists; semantics of DeltaVectorIndex.cs:95-121
 *      without the id-dedupe, which sharding makes unnecessary): parts x nq x k_in candidate lists
 *      -> nq x k_out, best first, ties to the lower part index.  rows < 0 mark empty slots. */
int pyrope_topk_merge_device(int64_t nq, int parts, int k_in, int k_out, const float *d_scores,
                             const int64_t *d_rows, float *d_scores_out, int64_t *d_rows_out,
                             int32_t *d_counts_out, void *stream);

/* The same with label de-duplication (dedupe != 0): a candidate whose row label already occurs in a LOWER part is
 * dropped — DeltaVectorIndex.cs:98-110's "one entry per id, the first list wins". */
int pyrope_topk_merge_dedupe_device(int64_t nq, int parts, int k_in, int k_out, const float *d_scores,
                                    const int64_t *d_rows, float *d_scores_out, int64_t *d_rows_out,
                                    int32_t *d_counts_out, int dedupe, void *stream);

/* ---- ONE index over the N GPUs of a box, one process (csrc/sharded.cu; SURVEY §8e "single process, 8 devices, one
 *      stream per device"): what a GpuVectorIndex constructed at Services/VectorIndexRegistry.cs:81-113 holds when
 *      the registry is configured with several devices.  One pyrope_index per device, one host thread per device.
 *      FLAT: rows dealt to the shards in consecutive blocks per add call (global row ordinals are the labels).
 *      IVF_*: every shard sees every row, Build keeps the inverted lists with list_id % N == shard; centroids and PQ
 *      codebooks are replicated (training is deterministic, the replicas agree bit for bit).
 *      Search: each shard ranks centroids for its slice of the batch and writes the probe lists into every peer's
 *      buffer over NVLink (peer stores + CUDA events, no host hop); every shard scans its lists for all queries, the
 *      IVF_PQ scan kernels exchange thresholds through peer memory while they run; local top-k lists land in device
 *      0's gather buffer and are merged there (one entry per row label).  Results equal the single-GPU index's.
 *      MaxScans (an insertion-/probe-order budget) cannot be split: max_scans >= 0 with N > 1 -> UNSUPPORTED.
 *      Errors: pyrope_sharded_last_error().  Calls on one handle are serialised internally. */
/* devices: n_devices CUDA ordinals, or NULL for 0..n_devices-1 (1 <= n_devices <= 8; peers must be NVLink/P2P reachable) */
int pyrope_sharded_create(int n_devices, const int *devices, int kind, int dim, int metric, int nlist, int pq_m,
                          int pq_k, pyrope_sharded **out);
int pyrope_sharded_destroy(pyrope_sharded *s);
int pyrope_sharded_device_count(pyrope_sharded *s, int *out);
/* the per-device index (and its CUDA ordinal) — for device-resident feeds: make that device current, then use the
 * pyrope_index_* calls; afterwards tell the sharded object the global row count with _note_rows */
int pyrope_sharded_shard(pyrope_sharded *s, int i, pyrope_index **index_out, int *device_out);
int pyrope_sharded_note_rows(pyrope_sharded *s, int64_t total_rows);
int pyrope_sharded_set_train_params(pyrope_sharded *s, int64_t max_train_rows, int max_iter);
int pyrope_sharded_set_codebooks(pyrope_sharded *s, int n_centroids, const float *centroids, const float *pq_codebooks);
/* IVectorIndex.Add for n rows (host pointers); labels NULL = global row ordinals; first_row_out = first ordinal */
int pyrope_sharded_add_batch(pyrope_sharded *s, int64_t n, const float *X, const int64_t *labels,
                             int64_t *first_row_out);
int pyrope_sharded_delete_row(pyrope_sharded *s, int64_t row);
/* IVectorIndex.Upsert of an existing row, semantics of pyrope_index_update_row.  FLAT: the owning shard's copy, in place
 * (un-deletes).  IVF_*: the row must be in the (replicated) write buffer and is updated on every shard; a list row ->
 * NOT_FOUND, shards that disagree -> INVALID_STATE. */
int pyrope_sharded_update_row(pyrope_sharded *s, int64_t row, const float *x);
/* pyrope_index_shadow_row on the shard owning the row's list (FLAT -> INVALID_STATE, no owner -> NOT_FOUND). */
int pyrope_sharded_shadow_row(pyrope_sharded *s, int64_t row, int shadowed);
/* pyrope_index_set_labels with global row ordinals (FLAT shards map their local rows through the row blocks). */
int pyrope_sharded_set_labels(pyrope_sharded *s, int64_t n_rows, const int64_t *labels_by_row);
int pyrope_sharded_build(pyrope_sharded *s);
/* pyrope_index_extend over N devices: every shard prepares on its own thread (assign, encode, merged lists), and the
 * merges are committed only if all of them prepared and all report the same set of buffered row ordinals (else
 * INVALID_STATE); on any failure no shard changes. */
int pyrope_sharded_extend(pyrope_sharded *s);
int pyrope_sharded_stats(pyrope_sharded *s, int64_t *live_rows_out);
/* read from the first shard: the replicas are bit-identical */
int pyrope_sharded_is_built(pyrope_sharded *s, int *out);
int pyrope_sharded_get_centroids(pyrope_sharded *s, float *centroids_out, int *n_out);
int pyrope_sharded_get_codebooks(pyrope_sharded *s, float *codebooks_out, int32_t *ksub_out);
/* IVectorIndex.Snapshot / Load over N devices.  `path` is a small binary manifest (shape, row count, the FLAT row blocks
 * and the names of the N shard files); shard i writes path.g<gen>.shard<i> with pyrope_index_snapshot, all in parallel,
 * the manifest is moved into place last and only then are the previous generation's shard files removed, so the
 * manifest on disk always names a complete set.  Load is all or nothing: the manifest is checked against the handle
 * (device count -> INVALID_ARG: no re-sharding on load, nor loading a single-device snapshot; kind / metric / m / k ->
 * INVALID_ARG, dim -> DIMENSION), every shard then parses and stages its file on its own thread (its shard identity
 * and row count must match the manifest), and the staged state is committed only when every shard succeeded; on any
 * failure the live index is left exactly as it was.  Missing file -> NOT_FOUND. */
int pyrope_sharded_snapshot(pyrope_sharded *s, const char *path);
int pyrope_sharded_load(pyrope_sharded *s, const char *path);
/* IVectorIndex.Search for nq queries over all shards: host buffers in / out (H2D of the queries to every device and
 * the D2H of the merged result inside the call). */
int pyrope_sharded_search_batch(pyrope_sharded *s, int64_t nq, const float *Q, int topk, int64_t max_scans,
                                int nprobe, float *scores_out, int64_t *rows_out, int32_t *counts_out);
/* the same with queries and outputs resident on the FIRST shard's device (the queries still travel to the peers) */
int pyrope_sharded_search_batch_device(pyrope_sharded *s, int64_t nq, const float *dQ_dev0, int topk,
                                       int64_t max_scans, int nprobe, float *d_scores_dev0, int64_t *d_rows_dev0,
                                       int32_t *d_counts_dev0);
/* device time (ms, CUDA events on the first shard's stream) of the most recent search: queries available -> merged result */
int pyrope_sharded_last_search_ms(pyrope_sharded *s, float *ms_out);
const char *pyrope_sharded_last_error(void);

/* ---- exchange over peer memory (csrc/peer.cu): the all-gather steps of a sharded search when every GPU has its own
 *      process (SURVEY §8e: local top-k lists, and the probe lists of a coarse stage split by query), written as peer
 *      stores over NVLink instead of a collective-library call.  One pyrope_peer_group per rank on that rank's current
 *      device; `slot_bytes` bounds one rank's contribution to one call, `n_slots` independent exchanges (<= 8) can be
 *      in use (e.g. slot 0 probes, 1 scores, 2 rows).  Every rank issues the same sequence of calls per slot.
 *      pyrope_peer_allgather_device enqueues, on `stream`: a copy of d_src (16-byte aligned, bytes_per_rank a multiple
 *      of 16) into every rank's buffer, a release of this call's epoch to the peers, and a wait for theirs; work
 *      enqueued after it on the same stream sees *d_gathered_out = [world][bytes_per_rank].  The area is double-buffered
 *      by call parity: consume the gathered data (on that stream) before the next-but-one call on the same slot.
 *      A rank whose peers never arrive faults after ~20 s instead of hanging the device.  Errors: pyrope_peer_last_error(). */
typedef struct pyrope_peer_group pyrope_peer_group;
int pyrope_peer_group_create(int world, int rank, size_t slot_bytes, int n_slots, pyrope_peer_group **out);
int pyrope_peer_group_destroy(pyrope_peer_group *g);
/* one process per GPU: exchange the 64-byte handles out of band (e.g. torch.distributed), then open all of them */
int pyrope_peer_group_handle(pyrope_peer_group *g, void *handle_out /* 64 bytes */);
int pyrope_peer_group_open(pyrope_peer_group *g, const void *handles /* world x 64 bytes, own entry ignored */);
/* one process, several GPUs (peer access enabled by the caller): hand over the peers' buffers directly */
int pyrope_peer_group_buffer(pyrope_peer_group *g, void **d_buffer_out);
int pyrope_peer_group_attach(pyrope_peer_group *g, void *const *buffers /* world entries, own entry ignored */);
int pyrope_peer_allgather_device(pyrope_peer_group *g, int slot, const void *d_src, size_t bytes_per_rank,
                                 const void **d_gathered_out, void *stream);
const char *pyrope_peer_last_error(void);

/* ---- Head+Tail on device: replaces DeltaVectorIndex (Vector/DeltaVectorIndex.cs) when BOTH sides are GPU
 *      indexes — a small mutable FLAT head and an IVF_FLAT / IVF_PQ / FLAT tail (VectorIndexRegistry.cs:110-111).
 *      Identity across the two sides is the row LABEL: the shim passes its id ordinal (Dictionary<string,long>) as
 *      the label of every row it adds to either side, so "same id" == "same label".  The delta object borrows the
 *      two handles (destroying it leaves them alive); writes keep going to the handles directly
 *      (Add/Upsert -> head, Delete -> both, DeltaVectorIndex.cs:26-74). */
/* DeltaVectorIndex..ctor :18-28: dimension / metric mismatch -> INVALID_ARG (ArgumentException). */
int pyrope_delta_create(pyrope_index *head, pyrope_index *tail, pyrope_delta **out);
/* The same with a tail sharded over the box's GPUs (IVF_FLAT / IVF_PQ only: a FLAT tail -> UNSUPPORTED; the head must
 * live on the tail's first device -> else INVALID_ARG).  Every pyrope_delta_* call accepts the result.  Search: the
 * head's top-k on its stream, the tail through the sharded search (cut to its own top k, as the reference asks the tail
 * for topK), then one de-duplicating merge; an IVF_PQ tail ignores MaxScans, an IVF_FLAT tail over N > 1 devices refuses
 * it (UNSUPPORTED); topk <= min(1024, 4096 / N).  Move: the head's live rows go to every shard's replica of the write
 * buffer (peer copies), the head is tombstoned only after every shard succeeded.  Snapshot: path.tail is the sharded
 * manifest of pyrope_sharded_snapshot. */
int pyrope_delta_create_sharded(pyrope_index *head, pyrope_sharded *tail, pyrope_delta **out);
int pyrope_delta_destroy(pyrope_delta *d);
/* DeltaVectorIndex.Search :76-122 for nq queries: head top-k and tail top-k with the SAME options (:85,88),
 * merged on the device — the head's copy of a label replaces the tail's, descending score, first topk.
 * One H2D of the queries, one D2H of the results, no host round trip between the stages.
 * topk <= 0 -> OUT_OF_RANGE (the FLAT head throws first, BruteForceVectorIndex.cs:278). */
int pyrope_delta_search_batch(pyrope_delta *d, int64_t nq, const float *Q, int topk, int64_t max_scans,
                              int nprobe, float *scores_out, int64_t *labels_out, int32_t *counts_out);
/* pyrope_delta_search_batch with topks[i] for query i: outputs have stride max(topks); row i holds counts[i] <= topks[i]
 * entries, equal to what pyrope_delta_search_batch over the same batch with topk = topks[i] returns for that query.
 * Head and tail are searched once at max(topks); the de-duplicating merge sees only the first topks[i] entries of
 * each side for query i, as the reference's Search with topK = topks[i] would.  Any topks[i] that the plain call
 * rejects fails the whole call with the same status. */
int pyrope_delta_search_batch_topk(pyrope_delta *d, int64_t nq, const float *Q, const int32_t *topks, int64_t max_scans,
                                   int nprobe, float *scores_out, int64_t *labels_out, int32_t *counts_out);
int pyrope_delta_search_batch_device(pyrope_delta *d, int64_t nq, const float *dQ, int topk,
                                     int64_t max_scans, int nprobe, float *d_scores, int64_t *d_labels,
                                     int32_t *d_counts, void *stream);
/* DeltaVectorIndex.Build :124-158 (compaction) without the per-vector Scan() -> Add loop: the head's live rows
 * move device-to-device, in scan order, into the tail's write buffer (a label the tail already buffers is
 * overwritten in place, one that sits in an inverted list is shadowed — Dictionary semantics of
 * IvfFlatVectorIndex.cs:47), every head row is tombstoned, then the tail is built.  moved_out = rows moved;
 * tail_rows_out (nullable, one entry per moved row in head scan order) = the tail row ordinal now holding it. */
int pyrope_delta_compact(pyrope_delta *d, int64_t *moved_out, int64_t *tail_rows_out);
/* The same in two calls: the move (head rows into the tail's buffer, head tombstoned) and the tail's Build.  A shim that
 * keeps id tables records tail_rows_out after the move whatever the build then returns, so a failed build (e.g. out of
 * memory while training) leaves every id addressable and can simply be retried. */
int pyrope_delta_move(pyrope_delta *d, int64_t *moved_out, int64_t *tail_rows_out);
int pyrope_delta_build_tail(pyrope_delta *d);
/* The Extend counterpart of pyrope_delta_build_tail (one-device and sharded tails): a compaction by Extend is
 * pyrope_delta_move followed by this call — the moved rows join the tail's lists without re-training. */
int pyrope_delta_extend_tail(pyrope_delta *d);
/* DeltaVectorIndex.GetStats :224-239: head count + tail count (duplicates counted twice, as there). */
int pyrope_delta_stats(pyrope_delta *d, int64_t *count_out);
/* DeltaVectorIndex.Snapshot / Load :160-222: path + ".head", path + ".tail" and a manifest at path. */
int pyrope_delta_snapshot(pyrope_delta *d, const char *path);
int pyrope_delta_load(pyrope_delta *d, const char *path);

/* ---- the reference's index classes with their STRING ids (csrc/vindex.cu): the host half of the drop-in.
 *      One pyrope_vindex is a BruteForceVectorIndex / IvfFlatVectorIndex / IvfPqVectorIndex (kind) or a
 *      DeltaVectorIndex over two of them; it keeps the id dictionaries those classes keep and maps their
 *      Add / Upsert / Delete / Build / Search semantics onto the row-ordinal entry points above, so the C# class
 *      behind IVectorIndex is a one-line forwarder per method.  Search returns id ORDINALS (process-wide, the
 *      row labels); pyrope_vindex_id turns one into its UTF-8 string.  Errors: pyrope_vindex_last_error().
 *      Status codes map to the exceptions the reference throws: INVALID_ARG -> ArgumentException ("Id cannot be
 *      empty."), DIMENSION -> ArgumentException("Vector dimension mismatch"), OUT_OF_RANGE ->
 *      ArgumentOutOfRangeException (FLAT topK <= 0), INVALID_STATE -> InvalidOperationException (FLAT duplicate
 *      Add, BruteForceVectorIndex.cs:141-144), NOT_FOUND -> FileNotFoundException (Load). */
int pyrope_vindex_create(int kind, int dim, int metric, int nlist, int pq_m, int pq_k, pyrope_vindex **out);
/* DeltaVectorIndex(head, tail) :18-28; head must be FLAT.  Borrows both (destroy the delta first). */
int pyrope_vindex_create_delta(pyrope_vindex *head, pyrope_vindex *tail, pyrope_vindex **out);
/* IvfFlatVectorIndex / IvfPqVectorIndex over n_devices GPUs (devices: CUDA ordinals or NULL for 0..n-1; IVF kinds only):
 * the row operations go to pyrope_sharded_*.  pyrope_vindex_create_delta takes it as the tail (with a FLAT head on
 * its first device); pyrope_vindex_native returns NULL for it. */
int pyrope_vindex_create_sharded(int n_devices, const int *devices, int kind, int dim, int metric, int nlist, int pq_m,
                                 int pq_k, pyrope_vindex **out);
int pyrope_vindex_destroy(pyrope_vindex *v);
int pyrope_vindex_native(pyrope_vindex *v, pyrope_index **out); /* row-ordinal handle (NULL for a delta or a sharded leaf) */
int pyrope_vindex_set_quantization(pyrope_vindex *v, int enable); /* BruteForceVectorIndex.EnableQuantization */
int pyrope_vindex_add(pyrope_vindex *v, const char *id, const float *vec, int len);
int pyrope_vindex_upsert(pyrope_vindex *v, const char *id, const float *vec, int len);
int pyrope_vindex_delete(pyrope_vindex *v, const char *id, int *removed_out);
int pyrope_vindex_build(pyrope_vindex *v); /* a delta compacts: DeltaVectorIndex.Build :124-158 */
/* Extend (pyrope_index_extend) with the id bookkeeping: buffered ids become list ids, shadowed list rows are gone, no id
 * is dropped (an IVF_PQ Build drops the ids it does not re-encode).  A delta compacts like pyrope_vindex_build with
 * pyrope_delta_extend_tail in place of the tail's Build; a FLAT tail -> UNSUPPORTED and an unbuilt tail -> INVALID_STATE
 * before any row moves. */
int pyrope_vindex_extend(pyrope_vindex *v);
/* nq queries of `len` floats each (len != Dimension -> DIMENSION). */
int pyrope_vindex_search(pyrope_vindex *v, int64_t nq, const float *Q, int len, int topk, int64_t max_scans,
                         int nprobe, float *scores_out, int64_t *id_ordinals_out, int32_t *counts_out);
int pyrope_vindex_id(int64_t id_ordinal, char *buf, int cap, int *len_out);
/* The same for a whole result list under ONE lock: the UTF-8 bytes of ids[0..n) are written back to back into buf
 * (at most cap bytes; call with buf = NULL to size it), offsets_out[i] .. offsets_out[i+1] delimit id i (n + 1 entries),
 * ordinals < 0 (empty result slots) give empty strings.  Id ordinals are reference counted and recycled once no index
 * holds the id any more, so results must be translated before the ids in them can be deleted — i.e. under the same
 * read lock the Search ran under, which is what the shim in INTEGRATION.md does. */
int pyrope_vindex_ids(const int64_t *id_ordinals, int64_t n, char *buf, int64_t cap, int64_t *offsets_out,
                      int64_t *bytes_out);
/* Size of the process-wide id table: ids currently held by some index, and ordinal slots ever allocated. */
int pyrope_vindex_id_table_size(int64_t *live_out, int64_t *slots_out);
int pyrope_vindex_stats(pyrope_vindex *v, int64_t *count_out, int *dim_out, int *metric_out);
int pyrope_vindex_get_centroids(pyrope_vindex *v, float *centroids_out, int *n_out); /* n_out 0 == null */
int pyrope_vindex_snapshot(pyrope_vindex *v, const char *path); /* index file(s) + "<file>.ids" id tables */
int pyrope_vindex_load(pyrope_vindex *v, const char *path);
const char *pyrope_vindex_last_error(void);

/* ---- data formats either side of the path (csrc/formats.cu; host only).  Errors: pyrope_formats_last_error().
 *      pyrope_parse_vector = VectorParsing.ParseVector (Utils/VectorParsing.cs:10-35): a VEC.ADD / VEC.SEARCH payload
 *      is tried as a JSON array, then as ',' / ' ' separated text, then taken as raw little-endian float32 (length a
 *      multiple of 4) — the binary form is what the benchmark client sends (VectorEncoding.ToLittleEndianBytes,
 *      Benchmarks/Encoding/VectorEncoding.cs:8-16 = pyrope_encode_vector).  Empty payload -> INVALID_ARG
 *      (ArgumentException), nothing matches -> INVALID_ARG "Unsupported vector format." (FormatException).
 *      n_out = element count; at most cap floats are written (call with out = NULL to size the buffer). */
int pyrope_parse_vector(const uint8_t *data, int64_t len, float *out, int64_t cap, int64_t *n_out);
int pyrope_encode_vector(const float *vec, int64_t n, uint8_t *out, int64_t cap_bytes);
/* FvecsReader.Read (Benchmarks/Datasets/FvecsReader.cs:14-60): records of int32 d + d float32.  limit < 0 = all
 * (null), 0 = none; skip = records to pass over first.  dimension <= 0 -> INVALID_ARG "Invalid vector dimension",
 * short record -> INVALID_ARG "Truncated fvecs record.", a torn 4-byte header at the end of the file ends the read.
 * out may be NULL to query count / dimension. */
int pyrope_fvecs_read(const char *path, int64_t limit, int64_t skip, float *out, int64_t cap_floats,
                      int64_t *count_out, int *dim_out);
/* The same records streamed into an index's device storage in 64 MiB batches (labels = row ordinals). */
int pyrope_index_add_fvecs(pyrope_index *h, const char *path, int64_t limit, int64_t *added_out);
const char *pyrope_formats_last_error(void);

/* ---- building blocks exposed for parity tests and for "next" rows (SURVEY §8f) --------------- */
/* KMeansUtils.FindNearestCentroid (KMeansUtils.cs:70-93), bit-exact: assign_out[i] = first index
 * of the best score.  Host pointers. */
int pyrope_coarse_assign(int metric, int dim, int64_t n, const float *X, int n_centroids,
                         const float *centroids, int32_t *assign_out);
/* KMeansUtils.Train (KMeansUtils.cs:10-68) on device, bit-exact w.r.t. the conventions in DESIGN.md.
 * data is n x dim with leading dimension ld.  Returns centroids (k_out rows) on the host. */
int pyrope_kmeans_train(int metric, int dim, int64_t n, int64_t ld, const float *data, int k,
                        int max_iter, int32_t seed, float *centroids_out, int *k_out,
                        int *iters_out);
/* ProductQuantizer.Encode (ProductQuantizer.cs:60-80), bit-exact.  codebooks [m][k][dim/m],
 * ksub [m] (NULL = k everywhere); X n x dim; codes_out n x m. */
int pyrope_pq_encode(int dim, int m, int k, const float *codebooks, const int32_t *ksub, int64_t n,
                     const float *X, uint8_t *codes_out);
/* ProductQuantizer.ComputeDistanceTable (ProductQuantizer.cs:98-120): table_out nq x m x k. */
int pyrope_pq_distance_table(int dim, int m, int k, const float *codebooks, int64_t nq,
                             const float *Q, float *table_out);
/* Fill a device buffer with uniform [0,1) fp32 from a counter-based generator (bench data for
 * configs too large for the sequential System.Random stream; documented in DESIGN.md). */
int pyrope_fill_uniform_device(float *d_out, int64_t n, uint64_t seed, uint64_t offset,
                               void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PYROPE_GPU_H */
