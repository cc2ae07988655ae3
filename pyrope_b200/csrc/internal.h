// internal.h — entry points the library's own modules call across files, not part of include/pyrope_gpu.h.  C linkage
// does not check that a prototype matches its definition, so the defining file and every caller include this header.
#pragma once

#include "../../include/pyrope_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

// ---- api.cu: Build, Extend and Load of one index in two halves, so that a sharded index can prepare every shard before
// it installs any.  _prepare_* stages the operation aside (the index is unchanged) and returns the staged state; _commit
// installs it and frees it, and cannot fail; _discard frees it unused.  All run with the index's device current.
typedef struct pyrope_internal_staged_info {
    int64_t n_moved;           // Build / Extend on a shard (shard world > 1): buffered row ordinals moving into the
    const int64_t* moved;      // lists (slot order), owned by the staged state
    int32_t shard_rank;        // Load: the shard identity and the rows ever added, as the file records them
    int32_t shard_world;
    int64_t next_row;
} pyrope_internal_staged_info;

int pyrope_internal_index_prepare_build(pyrope_index* h, void** staged_out, pyrope_internal_staged_info* info);
int pyrope_internal_index_prepare_extend(pyrope_index* h, void** staged_out, pyrope_internal_staged_info* info);
int pyrope_internal_index_prepare_load(pyrope_index* h, const char* path, void** staged_out, pyrope_internal_staged_info* info);
void pyrope_internal_index_commit(pyrope_index* h, void* staged);
void pyrope_internal_index_discard(void* staged);

// api.cu: rows ever added according to a snapshot's header (validates the magic only)
int pyrope_internal_snapshot_next_row(const char* path, int64_t* next_row_out);
// api.cu: the compaction's per-tail step of a Head+Tail whose tail is sharded, run on each shard's thread.  _reserve makes
// room for n more buffer rows before any shard writes; _absorb adds the rows (tail_absorb)
int pyrope_internal_tail_reserve(pyrope_index* tl, int64_t n);
int pyrope_internal_tail_absorb(pyrope_index* tl, int64_t n, const float* dX, const int64_t* dL, const int64_t* labels_host,
                                int64_t* tail_rows_out);
// api.cu: FLAT / IVF_FLAT / IVF_PQ of an index; the dimension of a Head+Tail and the largest topK its search accepts
int pyrope_internal_index_kind(pyrope_index* h, int* kind_out);
int pyrope_internal_delta_limits(pyrope_delta* d, int* dim_out, int* max_topk_out);

// ---- sharded.cu: rows ever added according to a sharded snapshot's manifest
int pyrope_internal_sharded_snapshot_next_row(const char* path, int64_t* next_row_out);
// sharded.cu: pyrope_sharded_search_batch_device whose shards first wait for q_ready (a cudaEvent_t, may be null)
int pyrope_internal_sharded_search_device(pyrope_sharded* s, int64_t nq, const float* dQ_dev0, int topk, int64_t max_scans,
                                          int nprobe, float* d_scores_dev0, int64_t* d_rows_dev0, int32_t* d_counts_dev0,
                                          void* q_ready);
// sharded.cu: the compaction's "_tail.Add per row" step on every shard of a sharded tail
int pyrope_internal_sharded_absorb(pyrope_sharded* s, int64_t n, const float* dX, const int64_t* dL, int src_device,
                                   const int64_t* labels_host, int64_t* tail_rows_out);

// ---- vindex.cu: the limits of a string-id index, and its search with a topK per query (the batcher's shim)
int pyrope_internal_vindex_limits(pyrope_vindex* v, int* dim_out, int* max_topk_out, int* nonpos_empty_out);
int pyrope_internal_vindex_search_topk(pyrope_vindex* v, int64_t nq, const float* Q, const int32_t* topks, int64_t max_scans,
                                       int nprobe, float* scores_out, int64_t* gids_out, int32_t* counts_out);

#ifdef __cplusplus
}
#endif
