// sharded.cu — ONE index over the N GPUs of a box, driven by one process (SURVEY §5 / §8e: "single process, 8 devices,
// one stream per device"), so that the C# class constructed at Services/VectorIndexRegistry.cs:81-113 gets N GPUs from
// one P/Invoke handle.  Built on the single-device entry points of include/pyrope_gpu.h:
//   * one pyrope_index per device, one persistent host thread per device (every CUDA call of a shard is issued with
//     that device current; N threads launch concurrently, so launch latency does not add up over the devices);
//   * FLAT: rows are dealt to the shards in consecutive blocks per add call, global row ordinals travel as labels;
//   * IVF_*: every shard sees every row and keeps the inverted lists with list_id % N == shard (pyrope_index_set_shard:
//     centroids and PQ codebooks replicated, training is deterministic so the replicas agree bit for bit);
//   * search: queries go to every device; shard r ranks centroids for ITS slice of the batch and writes the probe
//     lists straight into every peer's probe buffer over NVLink (peer stores, no host hop, no collective library),
//     CUDA events order the peers' streams; every shard scans its lists for all queries — the scan kernels exchange
//     per-query thresholds in flight through peer memory (pyrope_index_threshold_exchange_attach) — and writes its
//     local top-k into device 0's gather buffer; device 0 merges (labels de-duplicated: pre-build buffer rows live on
//     every shard) and returns the result.
// The merge semantics are DeltaVectorIndex.cs:95-121's: best score first, one entry per id.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <sys/stat.h>

#include <cuda_runtime.h>

#include "../../include/pyrope_gpu.h"
#include "internal.h"

namespace {

// reusable barrier for the worker threads of one job
struct HostBarrier {
    std::mutex mu;
    std::condition_variable cv;
    int n = 0, waiting = 0;
    uint64_t gen = 0;
    void wait() {
        std::unique_lock<std::mutex> g(mu);
        const uint64_t my = gen;
        if (++waiting == n) { waiting = 0; ++gen; cv.notify_all(); }
        else cv.wait(g, [&] { return gen != my; });
    }
};

struct Worker {
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, quit = false, done = true;
};

__global__ void scatter_words_kernel(const int64_t* __restrict__ src, int64_t n, int64_t* d0, int64_t* d1, int64_t* d2, int64_t* d3,
                                     int64_t* d4, int64_t* d5, int64_t* d6, int64_t* d7, int64_t off) {
    // one launch writes this shard's slice into every device's copy (peer stores over NVLink)
    int64_t* dst[8] = {d0, d1, d2, d3, d4, d5, d6, d7};
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t v = src[i];
#pragma unroll
    for (int p = 0; p < 8; ++p)
        if (dst[p]) dst[p][off + i] = v;
}

}  // namespace

struct pyrope_sharded {
    int n = 0, kind = 0, dim = 0, metric = 0, nlist = 0, m = 0, k = 0;
    std::vector<int> dev;
    std::vector<pyrope_index*> shard;
    std::vector<cudaStream_t> st;
    std::vector<cudaEvent_t> ev_probe, ev_res;
    std::vector<Worker*> workers;
    HostBarrier bar;
    std::mutex mu;  // one call at a time
    bool built = false, exchange = false;
    int64_t next_row = 0;
    // FLAT: where a global row lives (one segment per add call and shard)
    struct Seg { int64_t g0, n; int shard; int64_t local0; };
    std::vector<Seg> segs;
    std::vector<int64_t> shard_rows;  // FLAT: rows per shard so far
    int64_t snap_gen = 0;             // generation of the most recent snapshot written by this handle
    // per-device search buffers (grown on demand), device 0 also holds the gather / merged buffers
    struct Buf { void* p = nullptr; size_t bytes = 0; };
    std::vector<Buf> dQ, pr_local, pr_all, sc, rw, cn;
    Buf g_sc, g_rw, m_sc, m_rw, m_cn;
    void* hQ = nullptr; size_t hQ_bytes = 0;      // pinned staging: queries in, results out
    void* hOut = nullptr; size_t hOut_bytes = 0;
    int64_t thr_cap = 0;
    uint32_t epoch = 0;          // batch counter of the threshold exchange, the same on every shard
    std::vector<void*> thr_arr;  // every shard's published-threshold array (device pointers, peer-accessible)
    float last_ms = 0.f;
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;  // device 0: around one search (queries resident -> merged result)
};

namespace {

typedef pyrope_sharded S;

void worker_main(Worker* w, int device) {
    cudaSetDevice(device);
    for (;;) {
        std::function<void()> job;
        {
            std::unique_lock<std::mutex> g(w->mu);
            w->cv.wait(g, [&] { return w->has_job || w->quit; });
            if (w->quit) return;
            job = std::move(w->job);
            w->has_job = false;
        }
        job();
        {
            std::lock_guard<std::mutex> g(w->mu);
            w->done = true;
        }
        w->cv.notify_all();
    }
}

// run fn(r) on every shard's thread, wait for all; returns the first non-zero status, with the message its fn left on
// that shard's thread
int run_all(S* s, const std::function<int(int)>& fn) {
    std::vector<int> rc((size_t)s->n, 0);
    std::vector<std::string> msg((size_t)s->n);
    for (int r = 0; r < s->n; ++r) {
        Worker* w = s->workers[(size_t)r];
        {
            std::lock_guard<std::mutex> g(w->mu);
            w->job = [&, r] {
                rc[(size_t)r] = fn(r);
                if (rc[(size_t)r] != PYROPE_OK) msg[(size_t)r] = pyrope_last_error();
            };
            w->has_job = true;
            w->done = false;
        }
        w->cv.notify_all();
    }
    for (int r = 0; r < s->n; ++r) {
        Worker* w = s->workers[(size_t)r];
        std::unique_lock<std::mutex> g(w->mu);
        w->cv.wait(g, [&] { return w->done; });
    }
    for (int r = 0; r < s->n; ++r)
        if (rc[(size_t)r] != PYROPE_OK) return fail(rc[(size_t)r], "shard %d (device %d): %s", r, s->dev[(size_t)r], msg[(size_t)r].c_str());
    return PYROPE_OK;
}

int grow(S::Buf& b, size_t need) {  // on the current device
    if (need <= b.bytes) return PYROPE_OK;
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
    CK(cudaMalloc(&b.p, need));
    b.bytes = need;
    return PYROPE_OK;
}

int grow_pinned(void** p, size_t* have, size_t need) {
    if (need <= *have) return PYROPE_OK;
    if (*p) cudaFreeHost(*p);
    *p = nullptr;
    *have = 0;
    CK(cudaMallocHost(p, need));
    *have = need;
    return PYROPE_OK;
}

// Build, Extend or Load on every shard, all or nothing: prepare(r, &staged) stages shard r's operation on its own thread,
// then check() compares what the shards staged.  Only if every shard prepared and the check passed does every shard
// install its staged state; otherwise every staged state is dropped and every shard is left as it was.
int stage_all(S* s, const std::function<int(int, void**)>& prepare, const std::function<int()>& check) {
    std::vector<void*> staged((size_t)s->n, nullptr);
    int rc = run_all(s, [&](int r) -> int { return prepare(r, &staged[(size_t)r]); });
    if (rc == PYROPE_OK) rc = check();
    if (rc != PYROPE_OK) {
        run_all(s, [&](int r) -> int { pyrope_internal_index_discard(staged[(size_t)r]); return PYROPE_OK; });
        return rc;
    }
    run_all(s, [&](int r) -> int { pyrope_internal_index_commit(s->shard[(size_t)r], staged[(size_t)r]); return PYROPE_OK; });
    return PYROPE_OK;
}

// Build and Extend consume every shard's replica of the write buffer: they go ahead only if every shard moves the same
// buffered row ordinals into its lists
int stage_consuming(S* s, int (*prepare)(pyrope_index*, void**, pyrope_internal_staged_info*)) {
    std::vector<std::vector<int64_t>> moved((size_t)s->n);
    auto prep = [&](int r, void** staged) -> int {
        pyrope_internal_staged_info info{};
        TRY(prepare(s->shard[(size_t)r], staged, &info));
        moved[(size_t)r].assign(info.moved, info.moved + info.n_moved);
        std::sort(moved[(size_t)r].begin(), moved[(size_t)r].end());
        return PYROPE_OK;
    };
    auto same = [&]() -> int {
        for (size_t r = 1; r < moved.size(); ++r)
            if (moved[r] != moved[0])
                return fail(PYROPE_ERR_INVALID_STATE, "shard %zu and shard 0 would move different buffered rows (%zu vs %zu): the buffer replicas diverged",
                            r, moved[r].size(), moved[0].size());
        return PYROPE_OK;
    };
    return stage_all(s, prep, same);
}

}  // namespace

extern "C" {

int pyrope_sharded_create(int n_devices, const int* devices, int kind, int dim, int metric, int nlist, int pq_m, int pq_k,
                          pyrope_sharded** out) {
    if (!out) return fail(PYROPE_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    int have = 0;
    CK(cudaGetDeviceCount(&have));
    if (n_devices < 1 || n_devices > 8) return fail(PYROPE_ERR_INVALID_ARG, "n_devices must be 1..8");
    if (n_devices > have) return fail(PYROPE_ERR_INVALID_ARG, "%d devices requested, %d visible", n_devices, have);
    S* s = new (std::nothrow) S();
    if (!s) return fail(PYROPE_ERR_OOM, "out of host memory");
    s->n = n_devices; s->kind = kind; s->dim = dim; s->metric = metric; s->nlist = nlist; s->m = pq_m; s->k = pq_k;
    s->bar.n = n_devices;
    for (int r = 0; r < n_devices; ++r) {
        const int d = devices ? devices[r] : r;
        if (d < 0 || d >= have) { delete s; return fail(PYROPE_ERR_INVALID_ARG, "device %d does not exist", d); }
        s->dev.push_back(d);
    }
    const size_t N = (size_t)n_devices;
    s->shard.assign(N, nullptr); s->st.assign(N, nullptr); s->ev_probe.assign(N, nullptr); s->ev_res.assign(N, nullptr);
    s->dQ.resize(N); s->pr_local.resize(N); s->pr_all.resize(N); s->sc.resize(N); s->rw.resize(N); s->cn.resize(N);
    s->shard_rows.assign(N, 0);
    s->thr_arr.assign(N, nullptr);
    for (int r = 0; r < n_devices; ++r) {
        Worker* w = new Worker();
        w->th = std::thread(worker_main, w, s->dev[(size_t)r]);
        s->workers.push_back(w);
    }
    int rc = run_all(s, [&](int r) -> int {
        TRY(pyrope_gpu_init(s->dev[(size_t)r]));
        for (int p = 0; p < s->n; ++p) {  // NVLink peer access to every other shard's device
            if (p == r) continue;
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, s->dev[(size_t)r], s->dev[(size_t)p]));
            if (!can) return fail(PYROPE_ERR_UNSUPPORTED, "device %d cannot access device %d", s->dev[(size_t)r], s->dev[(size_t)p]);
            cudaError_t e = cudaDeviceEnablePeerAccess(s->dev[(size_t)p], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                return fail(PYROPE_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
            cudaGetLastError();
        }
        TRY(pyrope_index_create(kind, dim, metric, nlist, pq_m, pq_k, &s->shard[(size_t)r]));
        if (kind != PYROPE_FLAT && s->n > 1) TRY(pyrope_index_set_shard(s->shard[(size_t)r], r, s->n));
        CK(cudaStreamCreateWithFlags(&s->st[(size_t)r], cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&s->ev_probe[(size_t)r], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&s->ev_res[(size_t)r], cudaEventDisableTiming));
        if (r == 0) { CK(cudaEventCreate(&s->ev_t0)); CK(cudaEventCreate(&s->ev_t1)); }
        return PYROPE_OK;
    });
    if (rc != PYROPE_OK) { pyrope_sharded_destroy(s); return rc; }
    *out = s;
    return PYROPE_OK;
}

int pyrope_sharded_destroy(pyrope_sharded* s) {
    if (!s) return PYROPE_OK;
    if (!s->workers.empty()) {
        run_all(s, [&](int r) -> int {
            const size_t i = (size_t)r;
            if (s->st[i]) cudaStreamSynchronize(s->st[i]);
            if (s->shard[i]) pyrope_index_destroy(s->shard[i]);
            for (S::Buf* b : {&s->dQ[i], &s->pr_local[i], &s->pr_all[i], &s->sc[i], &s->rw[i], &s->cn[i]})
                if (b->p) cudaFree(b->p);
            if (r == 0) {
                for (S::Buf* b : {&s->g_sc, &s->g_rw, &s->m_sc, &s->m_rw, &s->m_cn})
                    if (b->p) cudaFree(b->p);
                if (s->hQ) cudaFreeHost(s->hQ);
                if (s->hOut) cudaFreeHost(s->hOut);
                if (s->ev_t0) cudaEventDestroy(s->ev_t0);
                if (s->ev_t1) cudaEventDestroy(s->ev_t1);
            }
            if (s->ev_probe[i]) cudaEventDestroy(s->ev_probe[i]);
            if (s->ev_res[i]) cudaEventDestroy(s->ev_res[i]);
            if (s->st[i]) cudaStreamDestroy(s->st[i]);
            return PYROPE_OK;
        });
    }
    for (Worker* w : s->workers) {
        {
            std::lock_guard<std::mutex> g(w->mu);
            w->quit = true;
        }
        w->cv.notify_all();
        if (w->th.joinable()) w->th.join();
        delete w;
    }
    delete s;
    return PYROPE_OK;
}

int pyrope_sharded_device_count(pyrope_sharded* s, int* out) {
    if (!s || !out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    *out = s->n;
    return PYROPE_OK;
}

int pyrope_sharded_shard(pyrope_sharded* s, int i, pyrope_index** index_out, int* device_out) {
    if (!s || i < 0 || i >= s->n) return fail(PYROPE_ERR_INVALID_ARG, "no such shard");
    if (index_out) *index_out = s->shard[(size_t)i];
    if (device_out) *device_out = s->dev[(size_t)i];
    return PYROPE_OK;
}

int pyrope_sharded_set_train_params(pyrope_sharded* s, int64_t max_train_rows, int max_iter) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    for (pyrope_index* h : s->shard) TRY(pyrope_index_set_train_params(h, max_train_rows, max_iter));
    return PYROPE_OK;
}

int pyrope_sharded_set_codebooks(pyrope_sharded* s, int n_centroids, const float* centroids, const float* pq_codebooks) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    std::lock_guard<std::mutex> g(s->mu);
    return run_all(s, [&](int r) -> int {
        TRY(pyrope_index_set_codebooks(s->shard[(size_t)r], n_centroids, centroids, pq_codebooks));
        return PYROPE_OK;
    });
}

// Rows added through the shard handles directly (device-resident feeds): tell the sharded object how many global rows exist.
int pyrope_sharded_note_rows(pyrope_sharded* s, int64_t total_rows) {
    if (!s || total_rows < 0) return fail(PYROPE_ERR_INVALID_ARG, "bad argument");
    s->next_row = total_rows;
    return PYROPE_OK;
}

int pyrope_sharded_add_batch(pyrope_sharded* s, int64_t n, const float* X, const int64_t* labels, int64_t* first_row_out) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    if (n < 0 || (n > 0 && !X)) return fail(PYROPE_ERR_INVALID_ARG, "vector is null");
    std::lock_guard<std::mutex> g(s->mu);
    const int64_t first = s->next_row;
    if (first_row_out) *first_row_out = first;
    if (n == 0) return PYROPE_OK;
    if (s->kind != PYROPE_FLAT) {
        // every shard sees every row (same row ordinals everywhere); Build keeps the lists a shard owns
        int rc = run_all(s, [&](int r) -> int {
            int64_t fr = -1;
            TRY(pyrope_index_add_batch(s->shard[(size_t)r], n, X, labels, &fr));
            if (fr != first) return fail(PYROPE_ERR_INVALID_STATE, "shard %d row ordinals diverged (%lld vs %lld)", r, (long long)fr, (long long)first);
            return PYROPE_OK;
        });
        if (rc == PYROPE_OK) s->next_row += n;
        return rc;
    }
    // FLAT: consecutive blocks, the global row ordinal (or the caller's label) is the row's label on its shard
    std::vector<int64_t> lab;
    if (!labels) {
        lab.resize((size_t)n);
        for (int64_t i = 0; i < n; ++i) lab[(size_t)i] = first + i;
        labels = lab.data();
    }
    std::vector<int64_t> local0((size_t)s->n, -1);
    int rc = run_all(s, [&](int r) -> int {
        const int64_t lo = n * r / s->n, hi = n * (r + 1) / s->n;
        if (hi > lo) TRY(pyrope_index_add_batch(s->shard[(size_t)r], hi - lo, X + (size_t)lo * s->dim, labels + lo, &local0[(size_t)r]));
        return PYROPE_OK;
    });
    if (rc != PYROPE_OK) return rc;
    for (int r = 0; r < s->n; ++r) {
        const int64_t lo = n * r / s->n, hi = n * (r + 1) / s->n;
        if (hi > lo) {
            s->segs.push_back({first + lo, hi - lo, r, local0[(size_t)r]});
            s->shard_rows[(size_t)r] += hi - lo;
        }
    }
    s->next_row += n;
    return PYROPE_OK;
}

int pyrope_sharded_delete_row(pyrope_sharded* s, int64_t row) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    std::lock_guard<std::mutex> g(s->mu);
    if (row < 0 || row >= s->next_row) return fail(PYROPE_ERR_NOT_FOUND, "row %lld not found", (long long)row);
    if (s->kind == PYROPE_FLAT) {
        for (const S::Seg& sg : s->segs)
            if (row >= sg.g0 && row < sg.g0 + sg.n) {
                const int rc = run_all(s, [&](int r) -> int {
                    return r == sg.shard ? pyrope_index_delete_row(s->shard[(size_t)r], sg.local0 + (row - sg.g0)) : PYROPE_OK;
                });
                return rc == PYROPE_ERR_NOT_FOUND ? fail(rc, "row not found") : rc;
            }
        return fail(PYROPE_ERR_NOT_FOUND, "row %lld not found", (long long)row);
    }
    // IVF: a buffered row lives on every shard, a list row on its owner only.  A shard without the row answers NOT_FOUND;
    // any other failure reaches the caller with that shard's message.
    std::vector<int> rcs((size_t)s->n, 0);
    const int rc = run_all(s, [&](int r) -> int {
        rcs[(size_t)r] = pyrope_index_delete_row(s->shard[(size_t)r], row);
        return rcs[(size_t)r] == PYROPE_ERR_NOT_FOUND ? PYROPE_OK : rcs[(size_t)r];
    });
    for (int c : rcs)
        if (c == PYROPE_OK) return PYROPE_OK;
    return rc != PYROPE_OK ? rc : fail(PYROPE_ERR_NOT_FOUND, "row %lld not found", (long long)row);
}

int pyrope_sharded_build(pyrope_sharded* s) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    std::lock_guard<std::mutex> g(s->mu);
    const int rc = stage_consuming(s, pyrope_internal_index_prepare_build);
    if (rc == PYROPE_OK && s->kind != PYROPE_FLAT) {
        int b = 0;
        pyrope_index_is_built(s->shard[0], &b);
        s->built = b != 0;
    }
    return rc;
}

int pyrope_sharded_extend(pyrope_sharded* s) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    if (s->kind == PYROPE_FLAT) return fail(PYROPE_ERR_UNSUPPORTED, "Extend needs an IVF index: FLAT has no inverted lists");
    std::lock_guard<std::mutex> g(s->mu);
    return stage_consuming(s, pyrope_internal_index_prepare_extend);
}

int pyrope_sharded_stats(pyrope_sharded* s, int64_t* live_rows_out) {
    if (!s || !live_rows_out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    int64_t tot = 0;
    for (int r = 0; r < s->n; ++r) {
        int64_t live = 0, buf = 0;
        TRY(pyrope_index_stats(s->shard[(size_t)r], &live, &buf, nullptr, nullptr));
        // IVF: buffered rows are replicated on every shard, list rows are not
        tot += (s->kind == PYROPE_FLAT || r == 0) ? live : live - buf;
    }
    *live_rows_out = tot;
    return PYROPE_OK;
}

// queries already on every device?  no: dQ_host / host outputs.  device_io != 0: Q is a DEVICE pointer on device 0 and the
// outputs are device pointers on device 0 (bench: HBM-resident timing); the queries still travel to the peers over NVLink.
// q_ready (device_io only, may be null): a CUDA event every shard waits for before it reads the queries.
static int sharded_search(S* s, int64_t nq, const float* Q, int topk, int64_t max_scans, int nprobe, float* scores_out,
                          int64_t* rows_out, int32_t* counts_out, int device_io, cudaEvent_t q_ready = nullptr) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    if (nq < 0 || (nq > 0 && !Q)) return fail(PYROPE_ERR_INVALID_ARG, "query is null");
    if (topk <= 0) {
        if (s->kind == PYROPE_FLAT) return fail(PYROPE_ERR_OUT_OF_RANGE, "topK must be positive.");
        for (int64_t i = 0; !device_io && i < nq; ++i) counts_out[i] = 0;
        return PYROPE_OK;
    }
    if (nq == 0) return PYROPE_OK;
    if (!scores_out || !rows_out || !counts_out) return fail(PYROPE_ERR_INVALID_ARG, "output buffer is null");
    if (max_scans >= 0 && s->n > 1)
        return fail(PYROPE_ERR_UNSUPPORTED, "MaxScans walks rows in insertion / probe order and cannot be split over devices");
    if ((int64_t)s->n * topk > 4096) return fail(PYROPE_ERR_UNSUPPORTED, "topK %d too large for %d shards", topk, s->n);
    std::lock_guard<std::mutex> g(s->mu);
    const int N = s->n, dim = s->dim, k = topk;
    const bool ivf = s->kind != PYROPE_FLAT;
    int built = 0;
    if (ivf) TRY(pyrope_index_is_built(s->shard[0], &built));
    const bool split = ivf && built && N > 1;
    const int P = nprobe >= 0 ? std::min(nprobe, std::max(s->nlist, 1)) : (s->kind == PYROPE_IVF_FLAT ? 3 : 1);
    const int64_t per = (nq + N - 1) / N;  // coarse slice per shard
    const size_t qbytes = sizeof(float) * (size_t)nq * dim;
    const bool use_thr = split && s->kind == PYROPE_IVF_PQ && P > 0;
    const bool thr_setup = use_thr && (!s->exchange || nq > s->thr_cap);
    const uint32_t epoch = ++s->epoch == 0 ? ++s->epoch : s->epoch;
    // Every shard's thread walks the same phases and meets the others at the same host barriers.  A failure must not
    // leave the peers waiting: it is recorded, the failing thread keeps walking (skipping the work), and so does
    // everybody else once they see the flag after the next barrier.
    std::atomic<bool> failed{false};
    int rc = run_all(s, [&](int r) -> int {
        const size_t i = (size_t)r;
        cudaStream_t st = s->st[i];
        int myrc = PYROPE_OK;
        std::string mymsg;
        auto phase = [&](const std::function<int()>& body) {
            if (failed.load() || myrc != PYROPE_OK) return;
            myrc = body();
            if (myrc != PYROPE_OK) { mymsg = pyrope_last_error(); failed.store(true); }
        };
        const size_t per_s = sizeof(float) * (size_t)nq * k, per_r = sizeof(int64_t) * (size_t)nq * k;
        // ---- phase 1: buffers, staging, threshold-exchange arrays
        phase([&]() -> int {
            TRY(grow(s->dQ[i], qbytes));
            TRY(grow(s->sc[i], per_s));
            TRY(grow(s->rw[i], per_r));
            TRY(grow(s->cn[i], sizeof(int32_t) * (size_t)nq));
            if (split) {
                TRY(grow(s->pr_local[i], sizeof(int64_t) * (size_t)per * P));
                TRY(grow(s->pr_all[i], sizeof(int64_t) * (size_t)per * N * P));
            }
            if (r == 0) {
                TRY(grow(s->g_sc, per_s * (size_t)N));
                TRY(grow(s->g_rw, per_r * (size_t)N));
                TRY(grow(s->m_sc, per_s));
                TRY(grow(s->m_rw, per_r));
                TRY(grow(s->m_cn, sizeof(int32_t) * (size_t)nq));
                if (!device_io) {
                    TRY(grow_pinned(&s->hQ, &s->hQ_bytes, qbytes));
                    TRY(grow_pinned(&s->hOut, &s->hOut_bytes, per_s + per_r + (size_t)nq * 4));
                    memcpy(s->hQ, Q, qbytes);
                }
            }
            if (thr_setup && s->exchange) TRY(pyrope_index_threshold_exchange_close(s->shard[i]));
            return PYROPE_OK;
        });
        s->bar.wait();  // nobody publishes into an array that is about to be replaced
        phase([&]() -> int {
            if (thr_setup) TRY(pyrope_index_threshold_exchange_array(s->shard[i], std::max<int64_t>(nq, 16384), &s->thr_arr[i]));
            return PYROPE_OK;
        });
        s->bar.wait();  // buffers and arrays of every shard exist (peers write into them), staging is filled
        // ---- phase 2: queries, coarse slice, probe lists to every peer
        phase([&]() -> int {
            if (thr_setup) TRY(pyrope_index_threshold_exchange_attach(s->shard[i], N, r, s->thr_arr.data()));
            if (use_thr) TRY(pyrope_index_threshold_exchange_epoch(s->shard[i], epoch));
            if (device_io) {
                if (q_ready) CK(cudaStreamWaitEvent(st, q_ready, 0));
                if (r == 0) { if (s->dQ[0].p != (const void*)Q) CK(cudaMemcpyAsync(s->dQ[0].p, Q, qbytes, cudaMemcpyDeviceToDevice, st)); }
                else CK(cudaMemcpyPeerAsync(s->dQ[i].p, s->dev[i], Q, s->dev[0], qbytes, st));
                if (r == 0) CK(cudaEventRecord(s->ev_t0, st));
            } else {
                if (r == 0) CK(cudaEventRecord(s->ev_t0, st));
                CK(cudaMemcpyAsync(s->dQ[i].p, s->hQ, qbytes, cudaMemcpyHostToDevice, st));
            }
            if (split) {
                const float* dQ = reinterpret_cast<const float*>(s->dQ[i].p);
                const int64_t qlo = std::min<int64_t>(nq, per * r), qhi = std::min<int64_t>(nq, qlo + per);
                int64_t* pl = reinterpret_cast<int64_t*>(s->pr_local[i].p);
                if (qhi > qlo) {
                    TRY(pyrope_index_coarse_probe_device(s->shard[i], qhi - qlo, dQ + (size_t)qlo * dim, P, pl, st));
                    int64_t* d[8] = {nullptr};
                    for (int p = 0; p < N; ++p) d[p] = reinterpret_cast<int64_t*>(s->pr_all[(size_t)p].p);
                    const int64_t words = (qhi - qlo) * P;
                    scatter_words_kernel<<<(unsigned)((words + 255) / 256), 256, 0, st>>>(pl, words, d[0], d[1], d[2], d[3], d[4], d[5],
                                                                                      d[6], d[7], qlo * P);
                    CK(cudaGetLastError());
                }
                CK(cudaEventRecord(s->ev_probe[i], st));
            }
            return PYROPE_OK;
        });
        s->bar.wait();  // every shard's probe event is recorded before anybody waits on it
        // ---- phase 3: scan, local top-k to the first shard's gather buffer
        phase([&]() -> int {
            const float* dQ = reinterpret_cast<const float*>(s->dQ[i].p);
            float* sc = reinterpret_cast<float*>(s->sc[i].p);
            int64_t* rw = reinterpret_cast<int64_t*>(s->rw[i].p);
            int32_t* cn = reinterpret_cast<int32_t*>(s->cn[i].p);
            if (split) {
                for (int p = 0; p < N; ++p)
                    if (p != r) CK(cudaStreamWaitEvent(st, s->ev_probe[(size_t)p], 0));
                TRY(pyrope_index_search_batch_probed_device(s->shard[i], nq, dQ, k, -1, P,
                                                            reinterpret_cast<const int64_t*>(s->pr_all[i].p), sc, rw, cn, st));
            } else {
                TRY(pyrope_index_search_batch_device(s->shard[i], nq, dQ, k, N > 1 ? -1 : max_scans, nprobe, sc, rw, cn, st));
            }
            if (r == 0) {
                CK(cudaMemcpyAsync(s->g_sc.p, sc, per_s, cudaMemcpyDeviceToDevice, st));
                CK(cudaMemcpyAsync(s->g_rw.p, rw, per_r, cudaMemcpyDeviceToDevice, st));
            } else {
                CK(cudaMemcpyPeerAsync((char*)s->g_sc.p + per_s * i, s->dev[0], sc, s->dev[i], per_s, st));
                CK(cudaMemcpyPeerAsync((char*)s->g_rw.p + per_r * i, s->dev[0], rw, s->dev[i], per_r, st));
            }
            CK(cudaEventRecord(s->ev_res[i], st));
            return PYROPE_OK;
        });
        s->bar.wait();  // every shard's result event is recorded
        // ---- phase 4: merge on the first shard's device
        phase([&]() -> int {
            if (r != 0) return PYROPE_OK;
            for (int p = 1; p < N; ++p) CK(cudaStreamWaitEvent(st, s->ev_res[(size_t)p], 0));
            float* ms = device_io ? scores_out : reinterpret_cast<float*>(s->m_sc.p);
            int64_t* mr = device_io ? rows_out : reinterpret_cast<int64_t*>(s->m_rw.p);
            int32_t* mc = device_io ? counts_out : reinterpret_cast<int32_t*>(s->m_cn.p);
            TRY(pyrope_topk_merge_dedupe_device(nq, N, k, k, reinterpret_cast<const float*>(s->g_sc.p),
                                                reinterpret_cast<const int64_t*>(s->g_rw.p), ms, mr, mc, ivf ? 1 : 0, st));
            if (!device_io) {
                char* ho = reinterpret_cast<char*>(s->hOut);
                CK(cudaMemcpyAsync(ho, ms, per_s, cudaMemcpyDeviceToHost, st));
                CK(cudaMemcpyAsync(ho + per_s, mr, per_r, cudaMemcpyDeviceToHost, st));
                CK(cudaMemcpyAsync(ho + per_s + per_r, mc, sizeof(int32_t) * (size_t)nq, cudaMemcpyDeviceToHost, st));
            }
            CK(cudaEventRecord(s->ev_t1, st));
            return PYROPE_OK;
        });
        cudaStreamSynchronize(st);  // the call is synchronous: every shard is idle when it returns
        s->bar.wait();               // ... and the first shard has consumed every peer's result
        if (myrc != PYROPE_OK) return fail(myrc, "%s", mymsg.c_str());
        return PYROPE_OK;
    });
    if (rc != PYROPE_OK) return rc;
    if (use_thr) { s->exchange = true; s->thr_cap = std::max<int64_t>(s->thr_cap, std::max<int64_t>(nq, 16384)); }
    if (!device_io) {
        const size_t per_s = sizeof(float) * (size_t)nq * k, per_r = sizeof(int64_t) * (size_t)nq * k;
        const char* ho = reinterpret_cast<const char*>(s->hOut);
        memcpy(scores_out, ho, per_s);
        memcpy(rows_out, ho + per_s, per_r);
        memcpy(counts_out, ho + per_s + per_r, sizeof(int32_t) * (size_t)nq);
    }
    cudaEventElapsedTime(&s->last_ms, s->ev_t0, s->ev_t1);
    return PYROPE_OK;
}

int pyrope_sharded_search_batch(pyrope_sharded* s, int64_t nq, const float* Q, int topk, int64_t max_scans, int nprobe,
                                float* scores_out, int64_t* rows_out, int32_t* counts_out) {
    return sharded_search(s, nq, Q, topk, max_scans, nprobe, scores_out, rows_out, counts_out, 0);
}

int pyrope_sharded_search_batch_device(pyrope_sharded* s, int64_t nq, const float* dQ_dev0, int topk, int64_t max_scans, int nprobe,
                                       float* d_scores_dev0, int64_t* d_rows_dev0, int32_t* d_counts_dev0) {
    return sharded_search(s, nq, dQ_dev0, topk, max_scans, nprobe, d_scores_dev0, d_rows_dev0, d_counts_dev0, 1);
}

int pyrope_sharded_last_search_ms(pyrope_sharded* s, float* ms_out) {
    if (!s || !ms_out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    *ms_out = s->last_ms;
    return PYROPE_OK;
}

// ---- Upsert / labels / codebooks: each call has the semantics of its pyrope_index_* namesake over the whole index

// FLAT: the segment holding a global row (nullptr if none)
static const S::Seg* flat_seg(const S* s, int64_t row) {
    for (const S::Seg& sg : s->segs)
        if (row >= sg.g0 && row < sg.g0 + sg.n) return &sg;
    return nullptr;
}

int pyrope_sharded_update_row(pyrope_sharded* s, int64_t row, const float* x) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    if (!x) return fail(PYROPE_ERR_INVALID_ARG, "vector is null");
    std::lock_guard<std::mutex> g(s->mu);
    if (row < 0 || row >= s->next_row) return fail(PYROPE_ERR_NOT_FOUND, "row %lld does not exist", (long long)row);
    if (s->kind == PYROPE_FLAT) {  // the owner's copy, in place (an Upsert un-deletes)
        const S::Seg* sg = flat_seg(s, row);
        if (!sg) return fail(PYROPE_ERR_NOT_FOUND, "row %lld does not exist", (long long)row);
        return run_all(s, [&](int r) -> int {
            if (r == sg->shard) TRY(pyrope_index_update_row(s->shard[(size_t)r], sg->local0 + (row - sg->g0), x));
            return PYROPE_OK;
        });
    }
    // IVF: only a buffered row can be updated, and the buffer is replicated: every shard must succeed
    std::vector<int> rcs((size_t)s->n, 0);
    const int rc = run_all(s, [&](int r) -> int { return rcs[(size_t)r] = pyrope_index_update_row(s->shard[(size_t)r], row, x); });
    int ok = 0;
    for (int c : rcs) ok += c == PYROPE_OK;
    if (ok == s->n) return PYROPE_OK;
    if (ok > 0) return fail(PYROPE_ERR_INVALID_STATE, "row %lld was updated on %d of %d shards", (long long)row, ok, s->n);
    return rcs[0] == PYROPE_ERR_NOT_FOUND ? fail(rcs[0], "row %lld is not in the write buffer", (long long)row) : rc;
}

int pyrope_sharded_shadow_row(pyrope_sharded* s, int64_t row, int shadowed) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    if (s->kind == PYROPE_FLAT) return fail(PYROPE_ERR_INVALID_STATE, "FLAT rows cannot be shadowed");
    std::lock_guard<std::mutex> g(s->mu);
    if (row < 0 || row >= s->next_row) return fail(PYROPE_ERR_NOT_FOUND, "row %lld not found", (long long)row);
    // a list row lives on the owner of its list only
    std::vector<int> rcs((size_t)s->n, 0);
    run_all(s, [&](int r) -> int { rcs[(size_t)r] = pyrope_index_shadow_row(s->shard[(size_t)r], row, shadowed); return PYROPE_OK; });
    for (int rc : rcs)
        if (rc == PYROPE_OK) return PYROPE_OK;
    return fail(PYROPE_ERR_NOT_FOUND, "row %lld is not in an inverted list", (long long)row);
}

int pyrope_sharded_set_labels(pyrope_sharded* s, int64_t n_rows, const int64_t* labels_by_row) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    std::lock_guard<std::mutex> g(s->mu);
    if (n_rows < s->next_row || (n_rows > 0 && !labels_by_row))
        return fail(PYROPE_ERR_INVALID_ARG, "labels for %lld rows needed, %lld given", (long long)s->next_row, (long long)n_rows);
    if (s->kind != PYROPE_FLAT)
        return run_all(s, [&](int r) -> int { TRY(pyrope_index_set_labels(s->shard[(size_t)r], n_rows, labels_by_row)); return PYROPE_OK; });
    // FLAT: a shard's local rows map back to global rows through the segment table
    return run_all(s, [&](int r) -> int {
        std::vector<int64_t> L((size_t)s->shard_rows[(size_t)r], -1);
        for (const S::Seg& sg : s->segs)
            if (sg.shard == r)
                for (int64_t i = 0; i < sg.n; ++i) L[(size_t)(sg.local0 + i)] = labels_by_row[(size_t)(sg.g0 + i)];
        TRY(pyrope_index_set_labels(s->shard[(size_t)r], (int64_t)L.size(), L.data()));
        return PYROPE_OK;
    });
}

// centroids and PQ codebooks are replicated bit for bit: read them from the first shard, on its thread
int pyrope_sharded_is_built(pyrope_sharded* s, int* out) {
    if (!s || !out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    TRY(pyrope_index_is_built(s->shard[0], out));
    return PYROPE_OK;
}

int pyrope_sharded_get_centroids(pyrope_sharded* s, float* centroids_out, int* n_out) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    std::lock_guard<std::mutex> g(s->mu);
    return run_all(s, [&](int r) -> int {
        if (r == 0) TRY(pyrope_index_get_centroids(s->shard[0], centroids_out, n_out));
        return PYROPE_OK;
    });
}

int pyrope_sharded_get_codebooks(pyrope_sharded* s, float* codebooks_out, int32_t* ksub_out) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    std::lock_guard<std::mutex> g(s->mu);
    return run_all(s, [&](int r) -> int {
        if (r == 0) TRY(pyrope_index_get_codebooks(s->shard[0], codebooks_out, ksub_out));
        return PYROPE_OK;
    });
}

}  // extern "C"

// ---- snapshot / load ----------------------------------------------------------------------------------------------
// `path` is a manifest; shard i's state is path.g<gen>.shard<i>, written by pyrope_index_snapshot on that shard's thread.
// The manifest is written last (tmp + rename) and the previous generation's shard files are removed only after that, so
// the manifest on disk always names a complete set of shard files.  Manifest, little-endian:
//   "PYRSHD01", int32 version, n, kind, dim, metric, nlist, m, k, int64 next_row, gen,
//   uint64 n_segs + n_segs x (int64 g0, int64 n, int32 shard, int64 local0)     (FLAT row blocks, none for IVF)
//   n x int64 shard_rows (FLAT), n x (uint32 name length, name, uint64 file bytes)   (names relative to the manifest)
namespace {

constexpr char kManifestMagic[8] = {'P', 'Y', 'R', 'S', 'H', 'D', '0', '1'};
constexpr int32_t kManifestVersion = 1;

struct Manifest {
    int32_t n = 0, kind = 0, dim = 0, metric = 0, nlist = 0, m = 0, k = 0;
    int64_t next_row = 0, gen = 0;
    std::vector<S::Seg> segs;
    std::vector<int64_t> shard_rows;
    std::vector<std::string> names;
    std::vector<uint64_t> bytes;
};

std::string dir_of(const std::string& path) {
    const size_t p = path.rfind('/');
    return p == std::string::npos ? std::string() : path.substr(0, p + 1);
}

bool file_bytes(const std::string& path, uint64_t* out) {
    struct stat st;
    if (stat(path.c_str(), &st) != 0) return false;
    *out = (uint64_t)st.st_size;
    return true;
}

// parse and check a manifest's own consistency; expect_n > 0: the shard count is checked right after the header (a
// manifest written by another device count is refused as such, before the rest of it is read)
int read_manifest(const char* path, Manifest& M, int expect_n = 0) {
    FILE* f = fopen(path, "rb");
    if (!f) return fail(PYROPE_ERR_NOT_FOUND, "Snapshot file not found: %s", path);
    bool ok = true;
    auto r = [&](void* p, size_t n) { if (ok && fread(p, 1, n, f) != n) ok = false; };
    auto rv32 = [&]() { int32_t v = 0; r(&v, 4); return v; };
    auto rv64 = [&]() { int64_t v = 0; r(&v, 8); return v; };
    char magic[8] = {0};
    r(magic, 8);
    int32_t version = rv32();
    if (!ok || memcmp(magic, kManifestMagic, 8) != 0 || version != kManifestVersion) {
        fclose(f);
        return fail(PYROPE_ERR_INVALID_ARG, "%s is not a sharded pyrope_gpu snapshot manifest", path);
    }
    M.n = rv32(); M.kind = rv32(); M.dim = rv32(); M.metric = rv32(); M.nlist = rv32(); M.m = rv32(); M.k = rv32();
    M.next_row = rv64(); M.gen = rv64();
    if (ok && expect_n > 0 && M.n != expect_n) {
        fclose(f);
        return fail(PYROPE_ERR_INVALID_ARG, "snapshot %s was written by %d shards, this index has %d devices (no re-sharding on load)",
                    path, M.n, expect_n);
    }
    const int64_t nsegs = rv64();
    ok = ok && M.n >= 1 && M.n <= 8 && M.next_row >= 0 && M.gen >= 1 && nsegs >= 0 && nsegs <= M.next_row;
    for (int64_t i = 0; ok && i < nsegs; ++i) {
        S::Seg sg;
        sg.g0 = rv64(); sg.n = rv64(); sg.shard = rv32(); sg.local0 = rv64();
        M.segs.push_back(sg);
    }
    for (int i = 0; ok && i < M.n; ++i) M.shard_rows.push_back(rv64());
    for (int i = 0; ok && i < M.n; ++i) {
        uint32_t len = 0;
        r(&len, 4);
        if (!ok || len == 0 || len > 4096) { ok = false; break; }
        std::string name(len, '\0');
        r(&name[0], len);
        uint64_t b = 0;
        r(&b, 8);
        if (name.find('/') != std::string::npos) ok = false;
        M.names.push_back(name);
        M.bytes.push_back(b);
    }
    fclose(f);
    if (!ok) return fail(PYROPE_ERR_INVALID_ARG, "corrupt or truncated snapshot manifest %s", path);
    // FLAT row blocks: inside [0, next_row) globally and inside their shard's local rows
    for (const S::Seg& sg : M.segs)
        if (sg.shard < 0 || sg.shard >= M.n || sg.n <= 0 || sg.g0 < 0 || sg.g0 + sg.n > M.next_row || sg.local0 < 0 ||
            sg.local0 + sg.n > M.shard_rows[(size_t)sg.shard])
            return fail(PYROPE_ERR_INVALID_ARG, "corrupt snapshot manifest %s: row block table", path);
    return PYROPE_OK;
}

}  // namespace

extern "C" {

int pyrope_sharded_snapshot(pyrope_sharded* s, const char* path) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    if (!path || !*path) return fail(PYROPE_ERR_INVALID_ARG, "Path cannot be empty");
    std::lock_guard<std::mutex> g(s->mu);
    const std::string base(path), dir = dir_of(base), stem = base.substr(dir.size());
    Manifest old;
    const bool have_old = read_manifest(path, old) == PYROPE_OK;
    // a generation that no manifest at this path names yet, so the files it writes replace none that are still referenced
    const int64_t gen = std::max(s->snap_gen, have_old ? old.gen : 0) + 1;
    std::vector<std::string> names((size_t)s->n);
    for (int r = 0; r < s->n; ++r) names[(size_t)r] = stem + ".g" + std::to_string(gen) + ".shard" + std::to_string(r);
    int rc = run_all(s, [&](int r) -> int { TRY(pyrope_index_snapshot(s->shard[(size_t)r], (dir + names[(size_t)r]).c_str())); return PYROPE_OK; });
    std::vector<uint64_t> bytes((size_t)s->n, 0);
    for (int r = 0; rc == PYROPE_OK && r < s->n; ++r)
        if (!file_bytes(dir + names[(size_t)r], &bytes[(size_t)r])) rc = fail(PYROPE_ERR_INVALID_STATE, "shard file %s vanished", names[(size_t)r].c_str());
    const std::string tmp = base + ".tmp";
    if (rc == PYROPE_OK) {
        FILE* f = fopen(tmp.c_str(), "wb");
        if (!f) {
            rc = fail(PYROPE_ERR_INVALID_ARG, "cannot open %s for writing", tmp.c_str());
        } else {
            bool ok = true;
            auto w = [&](const void* p, size_t n) { if (ok && fwrite(p, 1, n, f) != n) ok = false; };
            auto w32 = [&](int32_t v) { w(&v, 4); };
            auto w64 = [&](int64_t v) { w(&v, 8); };
            w(kManifestMagic, 8);
            w32(kManifestVersion); w32(s->n); w32(s->kind); w32(s->dim); w32(s->metric); w32(s->nlist); w32(s->m); w32(s->k);
            w64(s->next_row); w64(gen);
            w64((int64_t)s->segs.size());
            for (const S::Seg& sg : s->segs) { w64(sg.g0); w64(sg.n); w32(sg.shard); w64(sg.local0); }
            for (int r = 0; r < s->n; ++r) w64(s->shard_rows[(size_t)r]);
            for (int r = 0; r < s->n; ++r) {
                const uint32_t len = (uint32_t)names[(size_t)r].size();
                w(&len, 4);
                w(names[(size_t)r].data(), len);
                w(&bytes[(size_t)r], 8);
            }
            if (fclose(f) != 0 || !ok) rc = fail(PYROPE_ERR_INVALID_STATE, "short write to %s", tmp.c_str());
            else if (rename(tmp.c_str(), path) != 0) rc = fail(PYROPE_ERR_INVALID_STATE, "cannot move %s into place", tmp.c_str());
        }
    }
    if (rc != PYROPE_OK) {  // the manifest on disk (if any) still names the previous, complete set
        remove(tmp.c_str());
        for (const std::string& nm : names) remove((dir + nm).c_str());
        return rc;
    }
    s->snap_gen = gen;
    if (have_old)  // the previous generation is no longer referenced
        for (const std::string& nm : old.names)
            if (std::find(names.begin(), names.end(), nm) == names.end()) remove((dir + nm).c_str());
    return PYROPE_OK;
}

int pyrope_sharded_load(pyrope_sharded* s, const char* path) {
    if (!s) return fail(PYROPE_ERR_INVALID_ARG, "handle is null");
    if (!path || !*path) return fail(PYROPE_ERR_INVALID_ARG, "Path cannot be empty");
    std::lock_guard<std::mutex> g(s->mu);
    Manifest M;
    {
        const int rc = read_manifest(path, M, s->n);
        if (rc == PYROPE_ERR_INVALID_ARG) {  // a single-device snapshot has its own magic: say so
            FILE* f = fopen(path, "rb");
            char magic[8] = {0};
            const bool single = f && fread(magic, 1, 8, f) == 8 && memcmp(magic, "PYRGPU01", 8) == 0;
            if (f) fclose(f);
            if (single)
                return fail(PYROPE_ERR_INVALID_ARG, "%s is a single-device snapshot; a sharded index loads only a sharded manifest", path);
        }
        if (rc != PYROPE_OK) return rc;
    }
    if (M.kind != s->kind || M.metric != s->metric || M.m != s->m || M.k != s->k)
        return fail(PYROPE_ERR_INVALID_ARG, "snapshot is of a different index type");
    if (M.dim != s->dim) return fail(PYROPE_ERR_DIMENSION, "Vector dimension mismatch");
    if (s->kind != PYROPE_FLAT && !M.segs.empty()) return fail(PYROPE_ERR_INVALID_ARG, "corrupt snapshot manifest %s: row blocks on an IVF index", path);
    const std::string dir = dir_of(path);
    for (int r = 0; r < s->n; ++r) {
        const std::string f = dir + M.names[(size_t)r];
        uint64_t b = 0;
        if (!file_bytes(f, &b)) return fail(PYROPE_ERR_NOT_FOUND, "Snapshot file not found: %s", f.c_str());
        if (b != M.bytes[(size_t)r])
            return fail(PYROPE_ERR_INVALID_ARG, "shard file %s holds %llu bytes, the manifest recorded %llu", f.c_str(),
                        (unsigned long long)b, (unsigned long long)M.bytes[(size_t)r]);
    }
    // every shard parses and stages its file on its own thread; nothing is installed unless all of them succeed
    const int rc = stage_all(s, [&](int r, void** staged) -> int {
        pyrope_internal_staged_info info{};
        const std::string f = dir + M.names[(size_t)r];
        TRY(pyrope_internal_index_prepare_load(s->shard[(size_t)r], f.c_str(), staged, &info));
        // IVF shards carry their shard identity and the replicated row count; FLAT shards are plain indexes of their rows
        const bool ivf = s->kind != PYROPE_FLAT;
        const int want_rank = ivf ? r : 0, want_world = ivf ? s->n : 1;
        const int64_t want_rows = ivf ? M.next_row : M.shard_rows[(size_t)r];
        if (info.shard_rank != want_rank || info.shard_world != want_world || info.next_row != want_rows)
            return fail(PYROPE_ERR_INVALID_ARG, "%s is shard %d of %d with %lld rows, the manifest expects shard %d of %d with %lld rows",
                        f.c_str(), info.shard_rank, info.shard_world, (long long)info.next_row, want_rank, want_world,
                        (long long)want_rows);
        return PYROPE_OK;
    }, [] { return PYROPE_OK; });
    if (rc != PYROPE_OK) return rc;
    s->next_row = M.next_row;
    s->segs = M.segs;
    s->shard_rows = M.shard_rows;
    s->snap_gen = std::max(s->snap_gen, M.gen);
    int b = 0;
    pyrope_index_is_built(s->shard[0], &b);
    s->built = s->kind != PYROPE_FLAT && b != 0;
    return PYROPE_OK;
}

// ---- internal (not in the public header) ---------------------------------------------------------------------------

// rows ever added according to a sharded snapshot's manifest (the string-id layer sizes its id tables with it)
int pyrope_internal_sharded_snapshot_next_row(const char* path, int64_t* next_row_out) {
    Manifest M;
    const int rc = read_manifest(path, M);
    if (rc != PYROPE_OK) return rc;
    *next_row_out = M.next_row;
    return PYROPE_OK;
}

// pyrope_sharded_search_batch_device whose shards wait for q_ready (a cudaEvent_t, may be null) before reading the queries
int pyrope_internal_sharded_search_device(pyrope_sharded* s, int64_t nq, const float* dQ_dev0, int topk, int64_t max_scans,
                                          int nprobe, float* d_scores_dev0, int64_t* d_rows_dev0, int32_t* d_counts_dev0,
                                          void* q_ready) {
    return sharded_search(s, nq, dQ_dev0, topk, max_scans, nprobe, d_scores_dev0, d_rows_dev0, d_counts_dev0, 1,
                          (cudaEvent_t)q_ready);
}

// The compaction step of a Head+Tail whose tail is this (IVF) index: n rows (dX n x dim, dL labels: device memory on
// src_device; labels_host the same labels) join every shard's replica of the write buffer, each shard shadowing the
// list entries it owns with those labels.  Every shard makes room first, so an allocation failure leaves all of them
// unchanged; every shard must then report the same row ordinals.
int pyrope_internal_sharded_absorb(pyrope_sharded* s, int64_t n, const float* dX, const int64_t* dL, int src_device,
                                   const int64_t* labels_host, int64_t* tail_rows_out) {
    if (!s || n < 0) return fail(PYROPE_ERR_INVALID_ARG, "bad argument");
    if (s->kind == PYROPE_FLAT) return fail(PYROPE_ERR_UNSUPPORTED, "a sharded FLAT index cannot be a Head+Tail tail");
    if (n == 0) return PYROPE_OK;
    std::lock_guard<std::mutex> g(s->mu);
    const size_t N = (size_t)s->n, xb = sizeof(float) * (size_t)n * s->dim, lb = sizeof(int64_t) * (size_t)n;
    std::vector<void*> bx(N, nullptr), bl(N, nullptr);
    std::vector<std::vector<int64_t>> rows(N, std::vector<int64_t>((size_t)n, -1));
    int rc = run_all(s, [&](int r) -> int {
        const size_t i = (size_t)r;
        TRY(pyrope_internal_tail_reserve(s->shard[i], n));
        CK(cudaMalloc(&bx[i], xb));
        CK(cudaMalloc(&bl[i], lb));
        CK(cudaMemcpyPeerAsync(bx[i], s->dev[i], dX, src_device, xb, s->st[i]));
        CK(cudaMemcpyPeerAsync(bl[i], s->dev[i], dL, src_device, lb, s->st[i]));
        CK(cudaStreamSynchronize(s->st[i]));
        return PYROPE_OK;
    });
    if (rc == PYROPE_OK)
        rc = run_all(s, [&](int r) -> int {
            const size_t i = (size_t)r;
            TRY(pyrope_internal_tail_absorb(s->shard[i], n, (const float*)bx[i], (const int64_t*)bl[i], labels_host, rows[i].data()));
            return PYROPE_OK;
        });
    run_all(s, [&](int r) -> int {
        if (bx[(size_t)r]) cudaFree(bx[(size_t)r]);
        if (bl[(size_t)r]) cudaFree(bl[(size_t)r]);
        return PYROPE_OK;
    });
    if (rc != PYROPE_OK) return rc;
    for (size_t r = 1; r < N; ++r)
        if (rows[r] != rows[0]) return fail(PYROPE_ERR_INVALID_STATE, "shard %zu placed the moved rows at other row ordinals than shard 0", r);
    for (int64_t i = 0; i < n; ++i) s->next_row = std::max(s->next_row, rows[0][(size_t)i] + 1);
    if (tail_rows_out) memcpy(tail_rows_out, rows[0].data(), lb);
    return PYROPE_OK;
}

}  // extern "C"
