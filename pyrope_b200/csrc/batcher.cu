// batcher.cu — host micro-batcher in front of the batched searches.
//
// The reference drives the index ONE query per call: every Garnet session thread runs
// `index.Search(request.Vector, request.TopK, searchOptions)` under a read lock
// (Extensions/VectorCommandSet.cs:458, BruteForceVectorIndex.cs:282).  A GPU wants batches, so the
// P/Invoke shim's Search enqueues its query here and blocks; one dispatcher thread per target collects
// whatever arrived within max_wait_us (or max_batch queries, whichever first), groups requests with equal
// (MaxScans, NProbe, topK class), issues ONE batched search per group and wakes the callers.  The target is a
// one-device index, a sharded index, a Head+Tail or a string-id index.  Pure host code on top of the C ABI: no
// CUDA in this file.
//
// The topK class of a request is the smallest power of two >= topK, capped at the target's limit, so callers that
// ask for different topK share a launch at the cost of at most 2x in k.  A group is searched once at its largest
// topK: index and sharded searches order every list by (score, position or label), so that search's first k
// entries per query are the query's own top k; a Head+Tail merges with the per-query k instead
// (pyrope_delta_search_batch_topk), because cutting its merged list would refill a slot an id shared by head and
// tail freed.
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pyrope_gpu.h"
#include "internal.h"

namespace {

enum Target { kIndex, kSharded, kDelta, kVindex };

struct Request {
    const float* query;
    int topk;
    int k_class;
    int64_t max_scans;
    int nprobe;
    float* scores;
    int64_t* rows;
    int32_t* count;
    int status = 0;
    std::string error;
    bool done = false;
    std::chrono::steady_clock::time_point t_in;
};

thread_local std::string g_berr;

int bfail(int code, const char* msg) {
    g_berr = msg;
    return code;
}

}  // namespace

struct pyrope_batcher {
    Target target = kIndex;
    void* handle = nullptr;  // borrowed: pyrope_index / pyrope_sharded / pyrope_delta / pyrope_vindex
    int dim = 0, max_batch = 256, max_wait_us = 200;
    int max_topk = 1024;        // the target's own topK limit (UNSUPPORTED above it)
    bool nonpos_empty = false;  // topK <= 0: empty result (IVF) instead of OUT_OF_RANGE (FLAT, Head+Tail)
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    std::deque<Request*> queue;
    bool stop = false;
    int64_t n_batches = 0, n_queries = 0;
    std::thread worker;

    int k_class(int topk) const {
        int c = 1;
        while (c < topk) c <<= 1;
        return std::min(c, max_topk);
    }

    // one batched search; outputs have stride max(topks); on failure err holds the raising layer's message
    int search(int64_t nb, const float* Q, const int32_t* topks, int kmax, int64_t max_scans, int nprobe, float* S,
               int64_t* R, int32_t* C, std::string& err) {
        int rc = PYROPE_OK;
        switch (target) {
            case kIndex:
                rc = pyrope_index_search_batch((pyrope_index*)handle, nb, Q, kmax, max_scans, nprobe, S, R, C);
                if (rc) err = pyrope_last_error();
                break;
            case kSharded:
                rc = pyrope_sharded_search_batch((pyrope_sharded*)handle, nb, Q, kmax, max_scans, nprobe, S, R, C);
                if (rc) err = pyrope_sharded_last_error();
                break;
            case kDelta:
                rc = pyrope_delta_search_batch_topk((pyrope_delta*)handle, nb, Q, topks, max_scans, nprobe, S, R, C);
                if (rc) err = pyrope_last_error();
                break;
            case kVindex:
                rc = pyrope_internal_vindex_search_topk((pyrope_vindex*)handle, nb, Q, topks, max_scans, nprobe, S, R, C);
                if (rc) err = pyrope_vindex_last_error();
                break;
        }
        return rc;
    }

    void run() {
        std::vector<Request*> batch;
        std::vector<float> Q, S;
        std::vector<int64_t> R;
        std::vector<int32_t> C, K;
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            cv_work.wait(lk, [&] { return stop || !queue.empty(); });
            if (stop && queue.empty()) return;
            // let the batch fill: until max_wait_us after the oldest request arrived, or max_batch queued
            const auto deadline = queue.front()->t_in + std::chrono::microseconds(max_wait_us);
            cv_work.wait_until(lk, deadline, [&] { return stop || (int)queue.size() >= max_batch; });
            // take the requests that share the first one's options and topK class (others wait for the next round)
            batch.clear();
            const Request* f = queue.front();
            for (auto it = queue.begin(); it != queue.end() && (int)batch.size() < max_batch;) {
                Request* r = *it;
                if (r->k_class == f->k_class && r->max_scans == f->max_scans && r->nprobe == f->nprobe) {
                    batch.push_back(r);
                    it = queue.erase(it);
                } else {
                    ++it;
                }
            }
            const int nprobe = batch[0]->nprobe;
            const int64_t max_scans = batch[0]->max_scans;
            lk.unlock();
            const size_t nb = batch.size();
            int kmax = 1;
            K.resize(nb);
            for (size_t i = 0; i < nb; ++i) {
                K[i] = batch[i]->topk;
                kmax = std::max(kmax, batch[i]->topk);
            }
            const size_t kk = (size_t)kmax;
            Q.resize(nb * (size_t)dim);
            S.assign(nb * kk, 0.f);
            R.assign(nb * kk, -1);
            C.assign(nb, 0);
            for (size_t i = 0; i < nb; ++i) memcpy(&Q[i * (size_t)dim], batch[i]->query, sizeof(float) * (size_t)dim);
            std::string err;
            const int rc = search((int64_t)nb, Q.data(), K.data(), kmax, max_scans, nprobe, S.data(), R.data(), C.data(), err);
            for (size_t i = 0; i < nb; ++i) {
                Request* r = batch[i];
                r->status = rc;
                r->error = err;
                if (!rc) {
                    const int c = std::min(C[i], r->topk);
                    *r->count = c;
                    for (int j = 0; j < c; ++j) { r->scores[j] = S[i * kk + (size_t)j]; r->rows[j] = R[i * kk + (size_t)j]; }
                }
            }
            lk.lock();
            n_batches += 1;
            n_queries += (int64_t)nb;
            for (Request* r : batch) r->done = true;
            cv_done.notify_all();
        }
    }
};

namespace {

int start(Target t, void* handle, int dim, int max_topk, bool nonpos_empty, int max_batch, int max_wait_us,
          pyrope_batcher** out) {
    pyrope_batcher* b = new (std::nothrow) pyrope_batcher();
    if (!b) return bfail(PYROPE_ERR_OOM, "out of host memory");
    b->target = t;
    b->handle = handle;
    b->dim = dim;
    b->max_topk = max_topk;
    b->nonpos_empty = nonpos_empty;
    if (max_batch > 0) b->max_batch = max_batch;
    if (max_wait_us >= 0) b->max_wait_us = max_wait_us;
    b->worker = std::thread([b] { b->run(); });
    *out = b;
    return PYROPE_OK;
}

}  // namespace

extern "C" {

int pyrope_batcher_create(pyrope_index* h, int max_batch, int max_wait_us, pyrope_batcher** out) {
    if (!h || !out) return bfail(PYROPE_ERR_INVALID_ARG, "null argument");
    int dim = 0, kind = 0;
    int rc = pyrope_index_stats(h, nullptr, nullptr, &dim, nullptr);
    if (!rc) rc = pyrope_internal_index_kind(h, &kind);
    if (rc) return bfail(rc, pyrope_last_error());
    return start(kIndex, h, dim, 1024, kind != PYROPE_FLAT, max_batch, max_wait_us, out);
}

int pyrope_batcher_create_sharded(pyrope_sharded* s, int max_batch, int max_wait_us, pyrope_batcher** out) {
    if (!s || !out) return bfail(PYROPE_ERR_INVALID_ARG, "null argument");
    pyrope_index* s0 = nullptr;
    int n = 0, dim = 0, kind = 0;
    int rc = pyrope_sharded_device_count(s, &n);
    if (!rc) rc = pyrope_sharded_shard(s, 0, &s0, nullptr);
    if (rc) return bfail(rc, pyrope_sharded_last_error());
    rc = pyrope_index_stats(s0, nullptr, nullptr, &dim, nullptr);
    if (!rc) rc = pyrope_internal_index_kind(s0, &kind);
    if (rc) return bfail(rc, pyrope_last_error());
    return start(kSharded, s, dim, std::min(1024, 4096 / n), kind != PYROPE_FLAT, max_batch, max_wait_us, out);
}

int pyrope_batcher_create_delta(pyrope_delta* d, int max_batch, int max_wait_us, pyrope_batcher** out) {
    if (!d || !out) return bfail(PYROPE_ERR_INVALID_ARG, "null argument");
    int dim = 0, lim = 0;
    const int rc = pyrope_internal_delta_limits(d, &dim, &lim);
    if (rc) return bfail(rc, pyrope_last_error());
    return start(kDelta, d, dim, lim, false, max_batch, max_wait_us, out);
}

int pyrope_batcher_create_vindex(pyrope_vindex* v, int max_batch, int max_wait_us, pyrope_batcher** out) {
    if (!v || !out) return bfail(PYROPE_ERR_INVALID_ARG, "null argument");
    int dim = 0, lim = 0, empty = 0;
    const int rc = pyrope_internal_vindex_limits(v, &dim, &lim, &empty);
    if (rc) return bfail(rc, pyrope_vindex_last_error());
    return start(kVindex, v, dim, lim, empty != 0, max_batch, max_wait_us, out);
}

int pyrope_batcher_destroy(pyrope_batcher* b) {
    if (!b) return PYROPE_OK;
    {
        std::lock_guard<std::mutex> g(b->mu);
        b->stop = true;
    }
    b->cv_work.notify_all();
    if (b->worker.joinable()) b->worker.join();
    delete b;
    return PYROPE_OK;
}

int pyrope_batcher_search(pyrope_batcher* b, const float* query, int topk, int64_t max_scans, int nprobe,
                          float* scores_out, int64_t* rows_out, int32_t* count_out) {
    if (!b || !query || !scores_out || !rows_out || !count_out) return PYROPE_ERR_INVALID_ARG;
    *count_out = 0;
    // what the target's own search answers this caller alone, whatever the rest of the batch asks
    if (topk <= 0) return b->nonpos_empty ? PYROPE_OK : bfail(PYROPE_ERR_OUT_OF_RANGE, "topK must be positive.");
    if (topk > b->max_topk) {
        char msg[96];
        snprintf(msg, sizeof msg, "topK %d exceeds the supported maximum %d", topk, b->max_topk);
        return bfail(PYROPE_ERR_UNSUPPORTED, msg);
    }
    Request r;
    r.query = query; r.topk = topk; r.k_class = b->k_class(topk); r.max_scans = max_scans; r.nprobe = nprobe;
    r.scores = scores_out; r.rows = rows_out; r.count = count_out;
    r.t_in = std::chrono::steady_clock::now();
    std::unique_lock<std::mutex> lk(b->mu);
    if (b->stop) return PYROPE_ERR_INVALID_STATE;
    b->queue.push_back(&r);
    b->cv_work.notify_one();
    b->cv_done.wait(lk, [&] { return r.done; });
    lk.unlock();
    if (r.status) g_berr = r.error;
    return r.status;
}

const char* pyrope_batcher_last_error(void) { return g_berr.c_str(); }

int pyrope_batcher_stats(pyrope_batcher* b, int64_t* batches_out, int64_t* queries_out) {
    if (!b) return PYROPE_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(b->mu);
    if (batches_out) *batches_out = b->n_batches;
    if (queries_out) *queries_out = b->n_queries;
    return PYROPE_OK;
}

}  // extern "C"
