// api.cu — host side of libpyrope_gpu.so: index objects, storage in HBM, build pipeline, search
// orchestration and the C ABI declared in include/pyrope_gpu.h.
//
// HBM layout (one index, one GPU):
//   Segment (FLAT rows / IVF pre-build buffer): X[cap][dim] fp32 row-major, dead[cap] u8,
//     labels[cap] i64, norms[cap] fp32 (Cosine only).  Scan order = slot order.
//   IVF lists (IvfLists): off[nc+1] i64; entries list-major: payload[total][dim] fp32 (IVF_FLAT) or
//     payload[total][m] u8 (IVF_PQ), rows/labels[total] i64, dead[total] u8 (allocated on first delete),
//     norms (Cosine IVF_FLAT); centroids[nc][dim], cnorms[nc], codebook[m][k][dim/m] fp32 zero padded, ksub[m].
// Build, Extend and Load replace the lists (and Build / Load the trained quantisers) the same way: a *_prepare that only
// reads the index stages everything that can fail in a Staged, then install swaps it in and cannot fail.
#include <cub/cub.cuh>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include <unordered_map>
#include "../../include/pyrope_gpu.h"
#include "common.cuh"
#include "dotnet_random.h"
#include "internal.h"
#include "kernels.h"

using namespace pyrope;

static thread_local std::string g_err;  // the library's error message, one per thread (internal.h)

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

namespace {

int g_num_sms = 148;
bool g_inited = false;

int ensure_init() {
    if (g_inited) return PYROPE_OK;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    g_num_sms = prop.multiProcessorCount;
    g_inited = true;
    return PYROPE_OK;
}

// grow-only device buffer; owns its memory, so it moves but does not copy
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) {
            release();
            std::swap(p, o.p);
            std::swap(bytes, o.bytes);
        }
        return *this;
    }
    ~DevBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
    // ensure capacity; keep = preserve first keep_bytes
    int ensure(size_t need, size_t keep_bytes, cudaStream_t st, bool exact = false) {
        if (need <= bytes) return PYROPE_OK;
        size_t nb = exact ? need : std::max(need, bytes + bytes / 2);
        void* np = nullptr;
        cudaError_t e = cudaMalloc(&np, nb);
        if (e != cudaSuccess && nb > need) {
            cudaGetLastError();
            nb = need;
            e = cudaMalloc(&np, nb);
        }
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(PYROPE_ERR_OOM, "cudaMalloc(%zu bytes) failed: %s", nb, cudaGetErrorString(e));
        }
        if (p && keep_bytes) {
            CK(cudaMemcpyAsync(np, p, keep_bytes, cudaMemcpyDeviceToDevice, st));
            CK(cudaStreamSynchronize(st));
        }
        if (p) cudaFree(p);
        p = np;
        bytes = nb;
        return PYROPE_OK;
    }
    template <typename T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

struct Segment {
    int dim = 0;
    bool cosine = false;
    bool reuse_slots = false;  // Dictionary<,> semantics (IVF buffers) vs List<> (FLAT)
    int64_t nslots = 0, cap = 0, live = 0, ndead = 0;
    DevBuf X, dead, labels, norms;
    std::vector<uint8_t> dead_h;
    std::vector<int64_t> slot_row;    // IVF buffers only
    std::vector<int64_t> free_stack;  // LIFO, IVF buffers only

    int reserve(int64_t n, cudaStream_t st, bool exact) {
        if (n <= cap) return PYROPE_OK;
        int64_t nc = exact ? n : std::max<int64_t>(n, cap + cap / 2 + 1024);
        TRY(X.ensure((size_t)nc * dim * sizeof(float), (size_t)nslots * dim * sizeof(float), st, true));
        size_t old_dead = dead.bytes;
        TRY(dead.ensure((size_t)nc, (size_t)nslots, st, true));
        if (dead.bytes > old_dead)
            CK(cudaMemsetAsync(dead.as<uint8_t>() + nslots, 0, dead.bytes - (size_t)nslots, st));
        TRY(labels.ensure((size_t)nc * sizeof(int64_t), (size_t)nslots * sizeof(int64_t), st, true));
        if (cosine) TRY(norms.ensure((size_t)nc * sizeof(float), (size_t)nslots * sizeof(float), st, true));
        cap = nc;
        return PYROPE_OK;
    }
    bool tc_dirty = true;  // hi/lo split copies stale (row overwritten, deleted or slot re-used)
    void clear() {
        tc_dirty = true;
        nslots = live = ndead = 0;
        dead_h.clear();
        slot_row.clear();
        free_stack.clear();
    }
    void release() {
        clear();
        cap = 0;
        X.release();
        dead.release();
        labels.release();
        norms.release();
    }
};

struct Workspace {
    DevBuf queue, pairs_s, pairs_l, cpairs_s, cpairs_l, probes, probes_raw, probe_scores, probe_cnt, allow, qnorm,
        qhi, qlo, tcq, tcc,  // tensor-core path: split queries, candidate queues, counts
        q16, qbad,           // fp16 queries and the rows that do not fit fp16
        tcg, tct,            // two-pass threshold: group maxima, per-query tau
        q8,                  // SQ8: quantised queries
        hq, hs, hl, hc,      // h*: staging for the host-pointer entry point
        ctc,                 // query-stationary coarse probe scratch
        lm;                  // list-major IVF_PQ scan scratch
};

// tf32 hi/lo split + per-row proxy terms of one operand table (base rows or centroids)
struct TcOperand {
    DevBuf hi, lo, scale, bias, amax;
    int64_t rows_valid = 0;
    bool dirty = true;
    // fp16 copy for the one-term tensor passes (kernels.h: launch_tc_half): rows it covers, and whether every value lies
    // within the range those passes are proven for (read back once per rebuild)
    DevBuf h16, xabs;
    int64_t h16_rows = 0;
    bool h16_ok = false;
    void invalidate() { dirty = true; h16_rows = 0; }
};

// The inverted lists of an IVF index.  Entry i of list c sits at off_h[c] <= i < off_h[c + 1]; payload rows are dim * 4
// bytes (IVF_FLAT vectors) or m bytes (IVF_PQ codes).  dead[i]: bit 0 deleted, bit 1 shadowed by a buffered row; dead /
// dead_h stay empty until the first flag is set, ndead counts the flagged entries.
struct IvfLists {
    DevBuf off, rows, labels, payload, dead, norms;
    std::vector<int64_t> off_h;
    std::vector<uint8_t> dead_h;
    int64_t total = 0, ndead = 0, max_len = 0;
};

}  // namespace

struct pyrope_index {
    int kind = 0, dim = 0, metric = 0, nlist = 0, m = 0, k = 0, sub = 0;
    int device = 0;  // CUDA ordinal current at creation: every call on this index expects it current
    cudaStream_t stream = nullptr;
    cudaStream_t last_stream = nullptr;
    std::mutex mu;

    Segment seg;
    int64_t next_row = 0;

    // IVF state
    bool built = false;
    int nc = 0;
    DevBuf centroids, cnorms, codebook;
    IvfLists lists;  // replaced only by install
    // compacted view of the lists for MaxScans-budgeted IVF_FLAT searches (compact_lists)
    DevBuf bv_vecs, bv_labels, bv_norms, bv_off;
    uint64_t lists_version = 1, bv_version = 0;  // lists_version moves whenever lists or their dead flags change
    // shape of the most recent list-major IVF_PQ search (for pyrope_index_last_search_scanned)
    int64_t lm_nq = 0; int lm_P = 0, lm_k = 0;
    std::vector<int32_t> ksub;
    // list-major IVF_PQ with m < 16: the equivalent 16-table quantiser (kernels.h, IvfPqScanParams::lm_codebook) and the
    // codes repeated to 16 bytes per row; rebuilt lazily after the codebook / the lists were replaced
    DevBuf lm_cb16, lm_codes16;
    bool lm_cb16_ok = false, lm_codes16_ok = false;
    DevBuf pq_cmax;            // list-major IVF_PQ: max codeword norm per sub-quantiser of the table the scan reads
    bool pq_cmax_ok = false;   // reset whenever that table is rewritten
    bool frozen = false;  // codebooks supplied by the caller
    int64_t max_train_rows = 0;
    int max_iter = 0;
    int shard_rank = 0, shard_world = 1;

    // FLAT with EnableQuantization (BruteForceVectorIndex.cs:36-40): byte copy of the rows, X8[cap][dpad], and which rows
    // have one (rows written while the flag was off do not, :176-181, :209-214)
    bool sq8 = false;
    int dpad = 0;
    int64_t x8_cap = 0;
    DevBuf x8, qvalid8;

    // multi-GPU threshold exchange (list-major IVF_PQ): this rank's published array (peers write into it over NVLink)
    // and the peers' arrays opened through CUDA IPC
    DevBuf thr_pub;
    int64_t thr_cap = 0;
    std::vector<unsigned long long*> peer_thr;
    bool peer_ipc = false;        // peer arrays were opened through CUDA IPC (else: same-process device pointers)
    uint32_t thr_epoch = 0;       // batch counter of the exchange (every rank runs the same sequence of batches)
    bool thr_epoch_set = false;   // the caller named the next batch's epoch itself

    // row ordinal -> location: >=0 buffer slot, <=-2 list position (-2-pos), -1 gone
    std::vector<int64_t> row_loc;
    bool lists_loc_valid = true;

    Workspace ws;
    TcOperand tc_seg, tc_cent;
    int tc_mode = -1;  // -1 auto, 0 off, 1 force (PYROPE_FLAT_TC)
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t evk[2] = {nullptr, nullptr};  // around the dominant kernel of the last search
    cudaStream_t aux = nullptr;               // side stream of the list-major path (threshold seed)
    cudaEvent_t evf[2] = {nullptr, nullptr};  // fork / join
    bool ev_valid = false, evk_valid = false;
    const char* dom_kernel = "";
    int last_launches = 0;
    int pq_force_generic = 0;
    int pq_lm_mode = -1;  // PYROPE_PQ_LM: 0 = query-major kernels only
};

namespace {

typedef pyrope_index Index;

// ------------------------------------------------------------------------------------------
// segment writes
// ------------------------------------------------------------------------------------------
int seg_append(Index* h, int64_t n, const float* X, bool x_on_device, const int64_t* labels,
               bool labels_on_device, int64_t first_row) {
    Segment& s = h->seg;
    cudaStream_t st = h->stream;
    const size_t rowb = (size_t)s.dim * sizeof(float);
    const cudaMemcpyKind xk = x_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const cudaMemcpyKind lk = labels_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    int64_t i = 0;
    // Dictionary<,> re-uses freed slots LIFO before growing
    while (s.reuse_slots && i < n && !s.free_stack.empty()) {
        int64_t slot = s.free_stack.back();
        s.free_stack.pop_back();
        CK(cudaMemcpyAsync(s.X.as<float>() + slot * s.dim, X + i * s.dim, rowb, xk, st));
        if (labels) CK(cudaMemcpyAsync(s.labels.as<int64_t>() + slot, labels + i, sizeof(int64_t), lk, st));
        else CK(launch_iota64(s.labels.as<int64_t>() + slot, 1, first_row + i, st));
        CK(cudaMemsetAsync(s.dead.as<uint8_t>() + slot, 0, 1, st));
        if (s.cosine) CK(launch_row_norms_exact(s.X.as<float>() + slot * s.dim, 1, s.dim, s.dim, s.norms.as<float>() + slot, st));
        s.tc_dirty = true;
        s.dead_h[(size_t)slot] = 0;
        s.slot_row[(size_t)slot] = first_row + i;
        s.ndead--;
        s.live++;
        if (h->kind != PYROPE_FLAT) h->row_loc[(size_t)(first_row + i)] = slot;
        ++i;
    }
    const int64_t rest = n - i;
    if (rest > 0) {
        TRY(s.reserve(s.nslots + rest, st, false));
        const int64_t slot0 = s.nslots;
        CK(cudaMemcpyAsync(s.X.as<float>() + slot0 * s.dim, X + i * s.dim, rowb * (size_t)rest, xk, st));
        if (labels) CK(cudaMemcpyAsync(s.labels.as<int64_t>() + slot0, labels + i, sizeof(int64_t) * (size_t)rest, lk, st));
        else CK(launch_iota64(s.labels.as<int64_t>() + slot0, rest, first_row + i, st));
        if (s.cosine) CK(launch_row_norms_exact(s.X.as<float>() + slot0 * s.dim, rest, s.dim, s.dim, s.norms.as<float>() + slot0, st));
        s.dead_h.resize((size_t)(slot0 + rest), 0);
        if (h->kind != PYROPE_FLAT) {
            s.slot_row.resize((size_t)(slot0 + rest));
            for (int64_t j = 0; j < rest; ++j) {
                s.slot_row[(size_t)(slot0 + j)] = first_row + i + j;
                h->row_loc[(size_t)(first_row + i + j)] = slot0 + j;
            }
        }
        s.nslots += rest;
        s.live += rest;
    }
    CK(cudaStreamSynchronize(st));  // inputs are only borrowed for the duration of the call
    return PYROPE_OK;
}

// SQ8 copies of segment rows [slot0, slot0 + n): quantised if the flag is on, else marked as having none
int sq8_rows(Index* h, int64_t slot0, int64_t n) {
    if (h->kind != PYROPE_FLAT || (!h->sq8 && !h->x8.p) || n <= 0) return PYROPE_OK;
    Segment& s = h->seg;
    cudaStream_t st = h->stream;
    if (s.cap > h->x8_cap) {
        const size_t old_rows = (size_t)std::min<int64_t>(h->x8_cap, s.nslots);
        TRY(h->x8.ensure((size_t)s.cap * h->dpad, old_rows * h->dpad, st, true));
        const size_t old_q = h->qvalid8.bytes;
        TRY(h->qvalid8.ensure((size_t)s.cap, old_rows, st, true));
        if (h->qvalid8.bytes > old_q) CK(cudaMemsetAsync(h->qvalid8.as<uint8_t>() + old_rows, 0, h->qvalid8.bytes - old_rows, st));
        h->x8_cap = s.cap;
    }
    if (h->sq8)
        CK(launch_sq8_quantize(s.X.as<float>() + slot0 * s.dim, n, s.dim, s.dim, h->x8.as<uint8_t>() + slot0 * h->dpad, h->dpad,
                               h->qvalid8.as<uint8_t>() + slot0, st));
    else
        CK(cudaMemsetAsync(h->qvalid8.as<uint8_t>() + slot0, 0, (size_t)n, st));
    CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

// A *_device search may still be running on the caller's stream: every mutator waits for it before it touches rows,
// tombstones or tensor-core operands the scan reads (searches enqueued AFTER the mutation are ordered by the
// synchronisation each mutator ends with).
int wait_last_search(Index* h) {
    if (h->last_stream && h->last_stream != h->stream) CK(cudaStreamSynchronize(h->last_stream));
    return PYROPE_OK;
}

int add_common(Index* h, int64_t n, const float* X, bool dev, const int64_t* labels, int64_t* first_row_out) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (n < 0 || (n > 0 && !X)) return fail(PYROPE_ERR_INVALID_ARG, "vector is null");
    std::lock_guard<std::mutex> g(h->mu);
    TRY(wait_last_search(h));
    const int64_t first = h->next_row;
    if (first_row_out) *first_row_out = first;
    if (n == 0) return PYROPE_OK;
    if (h->kind != PYROPE_FLAT) h->row_loc.resize((size_t)(first + n), -1);
    h->next_row += n;
    const int64_t slot0 = h->seg.nslots;
    int r = seg_append(h, n, X, dev, labels, dev, first);
    if (r != PYROPE_OK) h->next_row = first;  // nothing was published
    else if (h->kind == PYROPE_FLAT) r = sq8_rows(h, slot0, n);
    return r;
}

int rebuild_row_loc(Index* h) {
    if (h->lists_loc_valid) return PYROPE_OK;
    std::fill(h->row_loc.begin(), h->row_loc.end(), (int64_t)-1);
    const IvfLists& L = h->lists;
    if (L.total > 0) {
        std::vector<int64_t> rows((size_t)L.total);
        CK(cudaMemcpy(rows.data(), L.rows.p, sizeof(int64_t) * rows.size(), cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < L.total; ++i)
            if (L.dead_h.empty() || !(L.dead_h[(size_t)i] & 1)) h->row_loc[(size_t)rows[(size_t)i]] = -2 - i;
    }
    for (int64_t s = 0; s < h->seg.nslots; ++s)
        if (!h->seg.dead_h[(size_t)s]) h->row_loc[(size_t)h->seg.slot_row[(size_t)s]] = s;
    h->lists_loc_valid = true;
    return PYROPE_OK;
}

int ensure_list_dead(Index* h) {
    IvfLists& L = h->lists;
    if (L.dead.p && L.dead_h.size() == (size_t)L.total) return PYROPE_OK;
    TRY(L.dead.ensure((size_t)std::max<int64_t>(L.total, 1), 0, h->stream, true));
    CK(cudaMemsetAsync(L.dead.p, 0, (size_t)std::max<int64_t>(L.total, 1), h->stream));
    L.dead_h.assign((size_t)L.total, 0);
    L.ndead = 0;
    return PYROPE_OK;
}

// Sets (set = true) or clears flag bits on the list entries at pos (ascending), keeping the host and device flags, the
// count of flagged entries and lists_version in step.  Caller synchronises the stream.
int set_list_flag(Index* h, const std::vector<int64_t>& pos, uint8_t bits, bool set) {
    if (pos.empty()) return PYROPE_OK;
    TRY(ensure_list_dead(h));
    IvfLists& L = h->lists;
    for (int64_t p : pos) {
        uint8_t& f = L.dead_h[(size_t)p];
        const uint8_t nv = set ? (f | bits) : (f & ~bits);
        L.ndead += (nv != 0) - (f != 0);
        f = nv;
    }
    h->lists_version++;
    const size_t lo = (size_t)pos.front(), n = (size_t)pos.back() + 1 - lo;
    CK(cudaMemcpyAsync(L.dead.as<uint8_t>() + lo, L.dead_h.data() + lo, n, cudaMemcpyHostToDevice, h->stream));
    return PYROPE_OK;
}

// ------------------------------------------------------------------------------------------
// training (KMeansUtils.Train on device)
// ------------------------------------------------------------------------------------------
__global__ void hist_kernel(const int32_t* a, int64_t n, unsigned long long* counts) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicAdd(&counts[a[i]], 1ull);
}
__global__ void iota32_kernel(int32_t* out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int32_t)i;
}
__global__ void widen_rows_kernel(const int32_t* order, const int64_t* src, int64_t n, int64_t* dst) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[order[i]];
}
__global__ void order_to_i64_kernel(const int32_t* order, int64_t n, int64_t* dst) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = order[i];
}

__global__ void shard_mask_kernel(int32_t* a, int64_t n, int nc, int rank, int world) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && (a[i] % world) != rank) a[i] = nc;  // parked in a dummy trailing cluster, dropped below
}

struct SortScratch {
    DevBuf keys_out, vals_in, vals_out, temp, counts, offs;
};

// stable sort of row indices by cluster id -> order[n], offs[nc+1] (device, int64)
int group_by_cluster(const int32_t* d_assign, int64_t n, int nc, SortScratch& sc, cudaStream_t st) {
    if (n >= (int64_t)1 << 31) return fail(PYROPE_ERR_UNSUPPORTED, "more than 2^31-1 rows per build");
    TRY(sc.keys_out.ensure(sizeof(int32_t) * (size_t)n, 0, st, true));
    TRY(sc.vals_in.ensure(sizeof(int32_t) * (size_t)n, 0, st, true));
    TRY(sc.vals_out.ensure(sizeof(int32_t) * (size_t)n, 0, st, true));
    TRY(sc.counts.ensure(sizeof(unsigned long long) * ((size_t)nc + 1), 0, st, true));
    TRY(sc.offs.ensure(sizeof(int64_t) * ((size_t)nc + 1), 0, st, true));
    iota32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sc.vals_in.as<int32_t>(), n);
    CK(cudaGetLastError());
    int end_bit = 1;
    while ((1ll << end_bit) < nc) ++end_bit;
    size_t tb = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, d_assign, sc.keys_out.as<int32_t>(), sc.vals_in.as<int32_t>(),
                                       sc.vals_out.as<int32_t>(), (int)n, 0, end_bit, st));
    size_t tb2 = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tb2, sc.counts.as<unsigned long long>(), sc.offs.as<unsigned long long>(),
                                     nc + 1, st));
    TRY(sc.temp.ensure(std::max(tb, tb2) + 16, 0, st, true));
    CK(cub::DeviceRadixSort::SortPairs(sc.temp.p, tb, d_assign, sc.keys_out.as<int32_t>(), sc.vals_in.as<int32_t>(),
                                       sc.vals_out.as<int32_t>(), (int)n, 0, end_bit, st));
    CK(cudaMemsetAsync(sc.counts.p, 0, sizeof(unsigned long long) * ((size_t)nc + 1), st));
    hist_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_assign, n, sc.counts.as<unsigned long long>());
    CK(cudaGetLastError());
    CK(cub::DeviceScan::ExclusiveSum(sc.temp.p, tb2, sc.counts.as<unsigned long long>(),
                                     sc.offs.as<unsigned long long>(), nc + 1, st));
    return PYROPE_OK;
}

// forward declaration (defined with the search helpers below)
int ensure_tc_operand(TcOperand& op, const float* X, int64_t n, int dim, int metric, const uint8_t* dead,
                      cudaStream_t st, const float* norms = nullptr);

struct AssignScratch {
    TcOperand cent;                       // tf32 split + proxy terms of the centroid table
    DevBuf qhi, qlo, tcq, tcc, flag, idx, nsel, temp, sub_assign, xg;
};

// KMeansUtils.FindNearestCentroid for n rows, bit-exact.  Small tables: exhaustive exact kernel.
// Large tables (>= 2048 centroids): tensor-core proxy scores shortlist k' = 17 centroids per row, the
// shortlist is re-evaluated in the reference's fp32 order (first index wins ties), and any row whose
// shortlist cannot be proven complete (its proxy spread within twice the proxy's and the reference's
// rounding bound, from |x| and the table's max |scale_c| |c|: assign_shortlist_kernel) is redone exhaustively.
int assign_rows(int metric, int dim, int64_t n, const float* X, int64_t ldx, int nc, const float* centroids,
                const float* cnorms, int32_t* assign, AssignScratch& sc, bool centroids_changed, cudaStream_t st) {
    if (n <= 0) return PYROPE_OK;
    const bool tc = nc >= 2048 && ldx == dim && flat_tc_supported(dim, 1) && !getenv("PYROPE_ASSIGN_EXACT");
    if (!tc) {
        CK(launch_assign_exact(metric, dim, n, X, ldx, nc, centroids, cnorms, assign, st));
        return PYROPE_OK;
    }
    if (centroids_changed) sc.cent.invalidate();
    TRY(ensure_tc_operand(sc.cent, centroids, nc, dim, metric, nullptr, st, cnorms));
    const int kprime = 1 + flat_tc_margin(1), cap = flat_tc_cap(kprime);
    const int64_t chunk = std::min<int64_t>(n, (int64_t)1 << 20);
    const int64_t chunk_pad = flat_tc_nq_pad(chunk);
    TRY(sc.qhi.ensure(sizeof(float) * (size_t)chunk * dim, 0, st, true));
    TRY(sc.qlo.ensure(sizeof(float) * (size_t)chunk * dim, 0, st, true));
    TRY(sc.tcq.ensure(sizeof(uint64_t) * (size_t)chunk_pad * cap, 0, st, true));
    TRY(sc.tcc.ensure(sizeof(int32_t) * (size_t)chunk_pad, 0, st, true));
    TRY(sc.flag.ensure((size_t)n, 0, st, true));
    for (int64_t c0 = 0; c0 < n; c0 += chunk) {
        const int64_t cn = std::min(chunk, n - c0);
        const float* Xc = X + (size_t)c0 * ldx;
        CK(launch_tc_prepare(Xc, cn, dim, metric, nullptr, sc.qhi.as<float>(), sc.qlo.as<float>(), nullptr, nullptr, 0, st));
        FlatTcParams tp{};
        tp.Q = Xc; tp.Qhi = sc.qhi.as<float>(); tp.Qlo = sc.qlo.as<float>(); tp.nq = cn; tp.dim = dim;
        tp.X = centroids; tp.Xhi = sc.cent.hi.as<float>(); tp.Xlo = sc.cent.lo.as<float>(); tp.n_rows = nc; tp.n_scan = nc;
        tp.scale = sc.cent.scale.as<float>(); tp.bias = sc.cent.bias.as<float>();
        tp.metric = metric; tp.k = 1; tp.kprime = kprime; tp.cap = cap; tp.splits = 1;
        tp.queue = sc.tcq.as<uint64_t>(); tp.counts = sc.tcc.as<int32_t>();
        CK(launch_flat_tc_select(tp, st));
        CK(launch_assign_from_shortlist(metric, dim, cn, Xc, ldx, centroids, cnorms, sc.cent.amax.as<float>(),
                                        sc.tcq.as<uint64_t>(), sc.tcc.as<int32_t>(), cap, kprime, assign + c0,
                                        sc.flag.as<uint8_t>() + c0, st));
    }
    // rows whose shortlist may be incomplete: redo exhaustively
    TRY(sc.idx.ensure(sizeof(int64_t) * (size_t)n, 0, st, true));
    TRY(sc.nsel.ensure(sizeof(int64_t), 0, st, true));
    size_t tb = 0;
    cub::CountingInputIterator<int64_t> iota(0);
    CK(cub::DeviceSelect::Flagged(nullptr, tb, iota, sc.flag.as<uint8_t>(), sc.idx.as<int64_t>(), sc.nsel.as<int64_t>(), n, st));
    TRY(sc.temp.ensure(tb + 16, 0, st, true));
    CK(cub::DeviceSelect::Flagged(sc.temp.p, tb, iota, sc.flag.as<uint8_t>(), sc.idx.as<int64_t>(), sc.nsel.as<int64_t>(), n, st));
    int64_t nsel = 0;
    CK(cudaMemcpyAsync(&nsel, sc.nsel.p, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (nsel > 0) {
        TRY(sc.xg.ensure(sizeof(float) * (size_t)nsel * dim, 0, st, true));
        TRY(sc.sub_assign.ensure(sizeof(int32_t) * (size_t)nsel, 0, st, true));
        CK(launch_gather_rows(X, (int64_t)dim * 4, sc.idx.as<int64_t>(), nsel, sc.xg.p, st));
        CK(launch_assign_exact(metric, dim, nsel, sc.xg.as<float>(), dim, nc, centroids, cnorms, sc.sub_assign.as<int32_t>(), st));
        CK(launch_scatter_i32(sc.sub_assign.as<int32_t>(), sc.idx.as<int64_t>(), nsel, assign, st));
    }
    return PYROPE_OK;
}

// KMeansUtils.Train: data n x dim (leading dimension ld) on device -> d_centroids [k][dim].
int kmeans_train_device(int metric, int dim, int64_t n, int64_t ld, const float* d_data, int k, int max_iter,
                        int32_t seed, float* d_centroids, int* k_out, int* iters_out, cudaStream_t st) {
    if (iters_out) *iters_out = 0;
    if (n == 0) { *k_out = 0; return PYROPE_OK; }
    if (k <= 0) k = 1;
    if (k > n) k = (int)n;
    *k_out = k;
    // init: data.OrderBy(_ => rnd.Next()).Take(k)
    std::vector<int64_t> init = kmeans_init_indices(n, k, seed);
    for (int c = 0; c < k; ++c)
        CK(cudaMemcpyAsync(d_centroids + (size_t)c * dim, d_data + (size_t)init[(size_t)c] * ld, sizeof(float) * dim,
                           cudaMemcpyDeviceToDevice, st));
    DevBuf assign, cn, changed;
    SortScratch sc;
    AssignScratch as;
    TRY(assign.ensure(sizeof(int32_t) * (size_t)n, 0, st, true));
    TRY(changed.ensure(sizeof(int), 0, st, true));
    if (metric == kCosine) TRY(cn.ensure(sizeof(float) * (size_t)k, 0, st, true));
    for (int it = 0; it < max_iter; ++it) {
        if (iters_out) *iters_out = it + 1;
        if (metric == kCosine) CK(launch_row_norms_exact(d_centroids, k, dim, dim, cn.as<float>(), st));
        TRY(assign_rows(metric, dim, n, d_data, ld, k, d_centroids, cn.as<float>(), assign.as<int32_t>(), as, true, st));
        TRY(group_by_cluster(assign.as<int32_t>(), n, k, sc, st));
        CK(cudaMemsetAsync(changed.p, 0, sizeof(int), st));
        CK(launch_kmeans_update(d_data, ld, dim, k, sc.offs.as<int64_t>(), sc.vals_out.as<int32_t>(), d_centroids,
                                changed.as<int>(), st));
        int ch = 0;
        CK(cudaMemcpyAsync(&ch, changed.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (!ch) break;
    }
    return PYROPE_OK;
}

// ------------------------------------------------------------------------------------------
// build
// ------------------------------------------------------------------------------------------
struct BuildData {
    const float* X = nullptr;  // [n][dim] device
    int64_t n = 0;
    DevBuf Xown, rows, labels;  // rows/labels per data row (device int64)
};

// Collect the rows a Build sees, in the reference's order: live list entries (list order) then
// live buffer slots (slot order).  IVF_PQ passes lists=false (IvfPqVectorIndex.cs:64).
int gather_build_data(const Index& h, bool include_lists, BuildData& bd) {
    cudaStream_t st = h.stream;
    const Segment& s = h.seg;
    const IvfLists& L = h.lists;
    const int dim = h.dim;
    // uniqueData (IvfFlatVectorIndex.cs:91-108) is a Dictionary filled from the lists first, then from the buffer:
    // an indexed id that was re-added through the buffer KEEPS its list position and takes the buffer's vector.
    // A shadowed list entry (flag 2) is matched to the live buffer slot carrying the same label; callers that do
    // not pass labels get the buffer row appended at the end instead (their labels differ by construction).
    std::unordered_map<int64_t, int64_t> repl_at;  // list position -> buffer slot that replaces it
    std::vector<uint8_t> slot_used;
    if (include_lists && h.built && !L.dead_h.empty() && s.live > 0) {
        std::vector<int64_t> sh;
        for (int64_t i = 0; i < L.total; ++i)
            if (L.dead_h[(size_t)i] == 2) sh.push_back(i);
        if (!sh.empty()) {
            DevBuf di, dl;
            TRY(di.ensure(sizeof(int64_t) * sh.size(), 0, st, true));
            TRY(dl.ensure(sizeof(int64_t) * sh.size(), 0, st, true));
            CK(cudaMemcpyAsync(di.p, sh.data(), sizeof(int64_t) * sh.size(), cudaMemcpyHostToDevice, st));
            CK(launch_gather_rows(L.labels.p, 8, di.as<int64_t>(), (int64_t)sh.size(), dl.p, st));
            std::vector<int64_t> shl(sh.size()), bl((size_t)s.nslots);
            CK(cudaMemcpyAsync(shl.data(), dl.p, sizeof(int64_t) * sh.size(), cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(bl.data(), s.labels.p, sizeof(int64_t) * (size_t)s.nslots, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            std::unordered_map<int64_t, int64_t> slot_of;
            for (int64_t i = 0; i < s.nslots; ++i)
                if (!s.dead_h[(size_t)i]) slot_of[bl[(size_t)i]] = i;
            slot_used.assign((size_t)s.nslots, 0);
            for (size_t j = 0; j < sh.size(); ++j) {
                auto it = slot_of.find(shl[j]);
                if (it == slot_of.end() || slot_used[(size_t)it->second]) continue;
                repl_at[sh[j]] = it->second;
                slot_used[(size_t)it->second] = 1;
            }
        }
    }
    std::vector<int64_t> list_pos;
    std::vector<int64_t> repl_out, repl_slot;  // output index <- buffer slot
    if (include_lists && h.built) {
        list_pos.reserve((size_t)L.total);
        for (int64_t i = 0; i < L.total; ++i) {
            if (L.dead_h.empty() || !L.dead_h[(size_t)i]) list_pos.push_back(i);
            else if (!repl_at.empty()) {
                auto it = repl_at.find(i);
                if (it == repl_at.end()) continue;
                repl_out.push_back((int64_t)list_pos.size());
                repl_slot.push_back(it->second);
                list_pos.push_back(i);
            }
        }
    }
    std::vector<int64_t> slots;
    const bool dense_buffer = (s.ndead == 0) && repl_out.empty();
    if (!dense_buffer) {
        slots.reserve((size_t)s.live);
        for (int64_t i = 0; i < s.nslots; ++i)
            if (!s.dead_h[(size_t)i] && (slot_used.empty() || !slot_used[(size_t)i])) slots.push_back(i);
    }
    const int64_t nb = dense_buffer ? s.nslots : (int64_t)slots.size();
    const int64_t nl = (int64_t)list_pos.size();
    bd.n = nl + nb;
    if (bd.n == 0) return PYROPE_OK;
    TRY(bd.rows.ensure(sizeof(int64_t) * (size_t)bd.n, 0, st, true));
    TRY(bd.labels.ensure(sizeof(int64_t) * (size_t)bd.n, 0, st, true));
    // rows of buffer slots come from the host map
    if (nl == 0 && dense_buffer) {
        bd.X = s.X.as<float>();  // zero-copy fast path
        CK(cudaMemcpyAsync(bd.rows.p, s.slot_row.data(), sizeof(int64_t) * (size_t)nb, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(bd.labels.p, s.labels.p, sizeof(int64_t) * (size_t)nb, cudaMemcpyDeviceToDevice, st));
        CK(cudaStreamSynchronize(st));
        return PYROPE_OK;
    }
    TRY(bd.Xown.ensure(sizeof(float) * (size_t)bd.n * dim, 0, st, true));
    bd.X = bd.Xown.as<float>();
    DevBuf idx;
    TRY(idx.ensure(sizeof(int64_t) * (size_t)std::max(nl, nb), 0, st, true));
    if (nl) {
        CK(cudaMemcpyAsync(idx.p, list_pos.data(), sizeof(int64_t) * (size_t)nl, cudaMemcpyHostToDevice, st));
        CK(launch_gather_rows(L.payload.p, (int64_t)dim * 4, idx.as<int64_t>(), nl, bd.Xown.p, st));
        CK(launch_gather_rows(L.rows.p, 8, idx.as<int64_t>(), nl, bd.rows.p, st));
        CK(launch_gather_rows(L.labels.p, 8, idx.as<int64_t>(), nl, bd.labels.p, st));
        CK(cudaStreamSynchronize(st));
    }
    if (!repl_out.empty()) {  // replaced entries: the buffer's vector and row ordinal at the list entry's place
        const int64_t nr = (int64_t)repl_out.size();
        DevBuf a, b, tx, tr;
        TRY(a.ensure(sizeof(int64_t) * (size_t)nr, 0, st, true));
        TRY(b.ensure(sizeof(int64_t) * (size_t)nr, 0, st, true));
        TRY(tx.ensure(sizeof(float) * (size_t)nr * dim, 0, st, true));
        TRY(tr.ensure(sizeof(int64_t) * (size_t)nr, 0, st, true));
        std::vector<int64_t> rrow((size_t)nr);
        for (int64_t i = 0; i < nr; ++i) rrow[(size_t)i] = s.slot_row[(size_t)repl_slot[(size_t)i]];
        CK(cudaMemcpyAsync(a.p, repl_slot.data(), sizeof(int64_t) * (size_t)nr, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(b.p, repl_out.data(), sizeof(int64_t) * (size_t)nr, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(tr.p, rrow.data(), sizeof(int64_t) * (size_t)nr, cudaMemcpyHostToDevice, st));
        CK(launch_gather_rows(s.X.p, (int64_t)dim * 4, a.as<int64_t>(), nr, tx.p, st));
        CK(launch_scatter_rows(tx.p, (int64_t)dim * 4, b.as<int64_t>(), nr, bd.Xown.p, st));
        CK(launch_scatter_rows(tr.p, 8, b.as<int64_t>(), nr, bd.rows.p, st));
        CK(cudaStreamSynchronize(st));
    }
    if (nb) {
        std::vector<int64_t> brow((size_t)nb);
        if (dense_buffer) {
            slots.resize((size_t)nb);
            for (int64_t i = 0; i < nb; ++i) slots[(size_t)i] = i;
        }
        for (int64_t i = 0; i < nb; ++i) brow[(size_t)i] = s.slot_row[(size_t)slots[(size_t)i]];
        CK(cudaMemcpyAsync(idx.p, slots.data(), sizeof(int64_t) * (size_t)nb, cudaMemcpyHostToDevice, st));
        CK(launch_gather_rows(s.X.p, (int64_t)dim * 4, idx.as<int64_t>(), nb, bd.Xown.as<float>() + (size_t)nl * dim, st));
        CK(launch_gather_rows(s.labels.p, 8, idx.as<int64_t>(), nb, bd.labels.as<int64_t>() + nl, st));
        CK(cudaMemcpyAsync(bd.rows.as<int64_t>() + nl, brow.data(), sizeof(int64_t) * (size_t)nb, cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
    }
    return PYROPE_OK;
}

// Stable grouping of n assigned rows by list (sc.vals_out = row order, sc.offs = [nc+1] offsets).  A shard keeps only
// the lists it owns (l % world == rank): rows of foreign lists sort to the tail and are cut off; kept_out = rows kept.
int group_rows(const Index& h, int32_t* d_assign, int64_t n, int nc, SortScratch& sc, int64_t* kept_out) {
    cudaStream_t st = h.stream;
    *kept_out = n;
    if (h.shard_world > 1) {
        shard_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_assign, n, nc, h.shard_rank, h.shard_world);
        CK(cudaGetLastError());
        TRY(group_by_cluster(d_assign, n, nc + 1, sc, st));
        CK(cudaMemcpyAsync(kept_out, sc.offs.as<int64_t>() + nc, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    } else {
        TRY(group_by_cluster(d_assign, n, nc, sc, st));
    }
    return PYROPE_OK;
}

// the write buffer is consumed by Build (IvfFlatVectorIndex.cs:143, IvfPqVectorIndex.cs:109) and by Extend;
// give large buffers back to the allocator, keep small ones for the next writes
void consume_buffer(Index* h) {
    if ((size_t)h->seg.cap * h->dim * sizeof(float) > ((size_t)256 << 20)) h->seg.release();
    else h->seg.clear();
}

// Staged::moved of a Build or an Extend: the row ordinals of the live buffer slots in slot order.  Only a shard of a
// sharded index needs them (every replica must move the same rows), so only a shard pays this host pass over the buffer
std::vector<int64_t> buffered_rows(const Index& h) {
    std::vector<int64_t> rows;
    if (h.shard_world == 1) return rows;
    const Segment& s = h.seg;
    rows.reserve((size_t)s.live);
    for (int64_t i = 0; i < s.nslots; ++i)
        if (!s.dead_h[(size_t)i]) rows.push_back(s.slot_row[(size_t)i]);
    return rows;
}

// What a Build, an Extend or a Load replaces in an index.  Its *_prepare fills it while only reading the index, and does
// everything that can fail there; install then swaps it in.
struct Staged {
    explicit Staged(const Index& h) : nc(h.nc), built(h.built), frozen(h.frozen) {}
    bool noop = true;  // an empty Build / Extend: nothing to install
    IvfLists lists;
    // quantiser: new centroids and (IVF_PQ) codebooks / ksub, from a Build that trains them or from a Load.  cnorms, when
    // present, replaces the centroid norms
    bool quantiser = false;
    DevBuf centroids, cnorms, codebook;
    std::vector<int32_t> ksub;
    int nc;
    bool built, frozen;
    // load: the write buffer and the counters the file holds replace the index's; otherwise the buffer moved into the
    // lists and is consumed (moved: its row ordinals in slot order, on a shard of a sharded index)
    bool load = false;
    Segment seg;
    int nlist = 0;
    int64_t next_row = 0;
    int32_t shard_rank = 0, shard_world = 1;
    std::vector<int64_t> moved;
};

// The only function that swaps trained state into an index, and the one place that resets what is derived from it.
// Cannot fail.  Caller holds h->mu.
void install(Index* h, Staged& S) {
    if (S.noop) return;
    h->lists = std::move(S.lists);
    h->lists_version++;
    h->lists_loc_valid = false;
    h->lm_codes16_ok = false;
    if (S.quantiser) {
        h->centroids = std::move(S.centroids);
        h->codebook = std::move(S.codebook);
        h->ksub.swap(S.ksub);
        h->lm_cb16_ok = false;
        h->pq_cmax_ok = false;
    }
    if (S.quantiser || S.cnorms.p) h->tc_cent.invalidate();
    if (S.cnorms.p) h->cnorms = std::move(S.cnorms);
    h->nc = S.nc;
    h->built = S.built;
    h->frozen = S.frozen;
    if (!S.load) {
        consume_buffer(h);
        return;
    }
    h->seg = std::move(S.seg);
    h->tc_seg.invalidate();
    h->nlist = S.nlist;
    h->next_row = S.next_row;
    h->shard_rank = S.shard_rank;
    h->shard_world = S.shard_world;
    if (h->kind != PYROPE_FLAT) h->row_loc.assign((size_t)h->next_row, -1);
    // SQ8 (FLAT): the reference's Load re-adds every row through InternalAdd (BruteForceVectorIndex.cs:93-97 ->
    // :162-184), which quantises it iff the LOADING index has EnableQuantization on at that moment — the flag is a
    // property of the object, not of the file.  Same here: with the flag on every loaded row gets its byte copy
    // (ScalarQuantizer is deterministic, so re-quantising reproduces the bytes the snapshotting index held), with it
    // off no loaded row has a quantised form (:312-322 keeps such rows invisible to a later quantised search).
    if (h->kind == PYROPE_FLAT && (h->sq8 || h->x8.p)) {
        h->x8_cap = 0;
        sq8_rows(h, 0, h->seg.nslots);  // best effort: the rows themselves are already in place
    }
}

// New lists in S.lists for the bd.n rows of a Build, assigned to nc lists; payload: one row of payload_row_bytes per row
int finish_lists(const Index& h, const BuildData& bd, int32_t* d_assign, int nc, const void* payload,
                 int64_t payload_row_bytes, Staged& S) {
    cudaStream_t st = h.stream;
    IvfLists& L = S.lists;
    SortScratch sc;
    int64_t n = bd.n;
    TRY(group_rows(h, d_assign, bd.n, nc, sc, &n));
    DevBuf order64;
    TRY(order64.ensure(sizeof(int64_t) * (size_t)bd.n, 0, st, true));
    order_to_i64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sc.vals_out.as<int32_t>(), n, order64.as<int64_t>());
    CK(cudaGetLastError());
    TRY(L.payload.ensure((size_t)std::max<int64_t>(n, 1) * (size_t)payload_row_bytes, 0, st, true));
    CK(launch_gather_rows(payload, payload_row_bytes, order64.as<int64_t>(), n, L.payload.p, st));
    TRY(L.rows.ensure(sizeof(int64_t) * (size_t)std::max<int64_t>(n, 1), 0, st, true));
    TRY(L.labels.ensure(sizeof(int64_t) * (size_t)std::max<int64_t>(n, 1), 0, st, true));
    widen_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sc.vals_out.as<int32_t>(), bd.rows.as<int64_t>(), n, L.rows.as<int64_t>());
    widen_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sc.vals_out.as<int32_t>(), bd.labels.as<int64_t>(), n, L.labels.as<int64_t>());
    CK(cudaGetLastError());
    TRY(L.off.ensure(sizeof(int64_t) * ((size_t)nc + 1), 0, st, true));
    CK(cudaMemcpyAsync(L.off.p, sc.offs.p, sizeof(int64_t) * ((size_t)nc + 1), cudaMemcpyDeviceToDevice, st));
    L.off_h.resize((size_t)nc + 1);
    CK(cudaMemcpyAsync(L.off_h.data(), sc.offs.p, sizeof(int64_t) * ((size_t)nc + 1), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    L.total = n;
    for (int c = 0; c < nc; ++c) L.max_len = std::max(L.max_len, L.off_h[(size_t)c + 1] - L.off_h[(size_t)c]);
    return PYROPE_OK;
}

// KMeansUtils.FindNearestCentroid against nc centroids (cnorms: their norms, read for Cosine) -> assign[n]
int assign_to_centroids(const Index& h, const float* centroids, const float* cnorms, int nc, const float* X, int64_t n,
                        DevBuf& assign) {
    cudaStream_t st = h.stream;
    TRY(assign.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(n, 1), 0, st, true));
    AssignScratch as;
    TRY(assign_rows(h.metric, h.dim, n, X, h.dim, nc, centroids, cnorms, assign.as<int32_t>(), as, true, st));
    CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

// rows of encoding work per residual chunk
int64_t pq_encode_chunk(int64_t n) { return std::min<int64_t>(n, (int64_t)4 << 20); }

// IvfPqVectorIndex.cs:82-90: residual to the assigned centroid, ProductQuantizer.Encode with the given codebooks
// (honouring ksub) -> codes[n][m].  res: scratch of at least pq_encode_chunk(n) rows (grown here if needed).
int pq_encode_rows(const Index& h, const float* centroids, const float* codebook, const std::vector<int32_t>& ksub,
                   const float* X, int64_t n, const int32_t* assign, DevBuf& res, DevBuf& codes) {
    cudaStream_t st = h.stream;
    const int dim = h.dim, m = h.m;
    const int64_t chunk = pq_encode_chunk(n);
    TRY(res.ensure(sizeof(float) * (size_t)std::max<int64_t>(chunk, 1) * dim, 0, st, true));
    DevBuf ksub_d;
    TRY(ksub_d.ensure(sizeof(int32_t) * (size_t)m, 0, st, true));
    CK(cudaMemcpyAsync(ksub_d.p, ksub.data(), sizeof(int32_t) * (size_t)m, cudaMemcpyHostToDevice, st));
    TRY(codes.ensure((size_t)std::max<int64_t>(n, 1) * m, 0, st, true));
    for (int64_t c0 = 0; c0 < n; c0 += chunk) {
        int64_t cn = std::min(chunk, n - c0);
        CK(launch_residuals(X + (size_t)c0 * dim, cn, dim, centroids, assign + c0, res.as<float>(), st));
        CK(launch_pq_encode_exact(res.as<float>(), cn, dim, m, h.k, codebook, ksub_d.as<int32_t>(),
                                  codes.as<uint8_t>() + (size_t)c0 * m, st));
    }
    CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

// ---- Build (IvfFlatVectorIndex.cs:87-143, IvfPqVectorIndex.cs:56-109): k-means over the rows Build sees trains new
// centroids (and, IVF_PQ, codebooks on the residuals) unless the caller froze them; every row is assigned, encoded and
// grouped into new lists.  IVF_FLAT sees its live list entries then its buffer, IVF_PQ its buffer alone (:64).
int build_prepare(const Index& h, Staged& S) {
    if (h.last_stream) CK(cudaStreamSynchronize(h.last_stream));
    if (h.kind == PYROPE_FLAT) return PYROPE_OK;  // BruteForceVectorIndex.cs:56
    cudaStream_t st = h.stream;
    const int dim = h.dim, m = h.m, K = h.k, sub = h.sub;
    const bool pq = h.kind == PYROPE_IVF_PQ;
    BuildData bd;
    TRY(gather_build_data(h, !pq, bd));
    const int64_t n = bd.n;
    if (n == 0) return PYROPE_OK;  // IvfFlatVectorIndex.cs:112, IvfPqVectorIndex.cs:62,65
    const int64_t ntrain = (h.max_train_rows > 0) ? std::min<int64_t>(h.max_train_rows, n) : n;
    if (!h.frozen) {
        int k = (int)std::min<int64_t>(h.nlist, n);
        if (k > ntrain) k = (int)ntrain;
        if (k <= 0) k = 1;
        TRY(S.centroids.ensure(sizeof(float) * (size_t)k * dim, 0, st, true));
        int iters = 0;
        TRY(kmeans_train_device(h.metric, dim, ntrain, dim, bd.X, k, h.max_iter > 0 ? h.max_iter : 10, pq ? 123 : 42,
                                S.centroids.as<float>(), &S.nc, &iters, st));
        S.quantiser = true;
    }
    const float* cent = (h.frozen ? h.centroids : S.centroids).as<float>();
    TRY(S.cnorms.ensure(sizeof(float) * (size_t)S.nc, 0, st, true));
    if (h.metric == kCosine) CK(launch_row_norms_exact(cent, S.nc, dim, dim, S.cnorms.as<float>(), st));
    DevBuf assign;
    TRY(assign_to_centroids(h, cent, S.cnorms.as<float>(), S.nc, bd.X, n, assign));
    const void* payload = bd.X;
    DevBuf res, codes;
    if (pq) {
        TRY(res.ensure(sizeof(float) * (size_t)std::max(pq_encode_chunk(n), h.frozen ? (int64_t)0 : ntrain) * dim, 0, st, true));
        if (!h.frozen) {  // PQ training on the residuals of the training rows (ProductQuantizer.cs:28-58)
            CK(launch_residuals(bd.X, ntrain, dim, cent, assign.as<int32_t>(), res.as<float>(), st));
            TRY(S.codebook.ensure(sizeof(float) * (size_t)m * K * sub, 0, st, true));
            CK(cudaMemsetAsync(S.codebook.p, 0, sizeof(float) * (size_t)m * K * sub, st));
            S.ksub.assign((size_t)m, 0);
            DevBuf cb1;
            TRY(cb1.ensure(sizeof(float) * (size_t)K * sub, 0, st, true));
            for (int mi = 0; mi < m; ++mi) {
                int kk = 0, iters = 0;
                TRY(kmeans_train_device(kL2, sub, ntrain, dim, res.as<float>() + (size_t)mi * sub, K, 10, 42 + mi,
                                        cb1.as<float>(), &kk, &iters, st));
                S.ksub[(size_t)mi] = kk;
                CK(cudaMemcpyAsync(S.codebook.as<float>() + (size_t)mi * K * sub, cb1.p, sizeof(float) * (size_t)kk * sub,
                                   cudaMemcpyDeviceToDevice, st));
                CK(cudaStreamSynchronize(st));
            }
        }
        TRY(pq_encode_rows(h, cent, (h.frozen ? h.codebook : S.codebook).as<float>(), h.frozen ? h.ksub : S.ksub, bd.X, n,
                           assign.as<int32_t>(), res, codes));
        payload = codes.p;
    }
    TRY(finish_lists(h, bd, assign.as<int32_t>(), S.nc, payload, pq ? m : (int64_t)dim * 4, S));
    IvfLists& L = S.lists;
    if (!pq && h.metric == kCosine) {
        TRY(L.norms.ensure(sizeof(float) * (size_t)std::max<int64_t>(L.total, 1), 0, st, true));
        CK(launch_row_norms_exact(L.payload.as<float>(), L.total, dim, dim, L.norms.as<float>(), st));
    }
    CK(cudaStreamSynchronize(st));
    S.built = true;
    S.moved = buffered_rows(h);
    S.noop = false;
    return PYROPE_OK;
}

// ---- Extend: append the write buffer to the inverted lists of a built IVF index without re-training.  Every live
// buffer row (slot order) goes to its nearest CURRENT centroid (assign_rows, as Build), IVF_PQ rows are encoded with the
// CURRENT codebooks, and each row is appended to the end of its list (rows of one list keep slot order: group_rows is a
// stable sort).  Old entries keep their order, row ordinals, labels and dead flags, except that shadowed entries (flag 2:
// their replacement has just left the buffer) become deleted.  A shard appends only to the lists it owns.
int extend_prepare(const Index& h, Staged& S) {
    if (h.kind == PYROPE_FLAT) return fail(PYROPE_ERR_UNSUPPORTED, "Extend needs an IVF index: FLAT has no inverted lists");
    if (!h.built) return fail(PYROPE_ERR_INVALID_STATE, "Extend needs a built index: call Build first");
    cudaStream_t st = h.stream;
    CK(cudaStreamSynchronize(st));
    if (h.last_stream) CK(cudaStreamSynchronize(h.last_stream));
    const Segment& s = h.seg;
    if (s.live == 0) return PYROPE_OK;
    const IvfLists& O = h.lists;
    IvfLists& L = S.lists;
    const int dim = h.dim, nc = h.nc;
    BuildData bd;
    TRY(gather_build_data(h, false, bd));  // live buffer slots, slot order
    const int64_t n = bd.n;
    DevBuf assign, res, codes, nnorm;
    TRY(assign_to_centroids(h, h.centroids.as<float>(), h.cnorms.as<float>(), nc, bd.X, n, assign));
    const bool pq = h.kind == PYROPE_IVF_PQ, cos_norms = !pq && h.metric == kCosine;
    const int64_t rb = pq ? h.m : (int64_t)dim * 4;
    if (pq) TRY(pq_encode_rows(h, h.centroids.as<float>(), h.codebook.as<float>(), h.ksub, bd.X, n, assign.as<int32_t>(), res, codes));
    if (cos_norms) {
        TRY(nnorm.ensure(sizeof(float) * (size_t)n, 0, st, true));
        CK(launch_row_norms_exact(bd.X, n, dim, dim, nnorm.as<float>(), st));
    }
    SortScratch sc;
    int64_t kept = 0;
    TRY(group_rows(h, assign.as<int32_t>(), n, nc, sc, &kept));
    std::vector<int64_t> offs_new((size_t)nc + 1);
    CK(cudaMemcpyAsync(offs_new.data(), sc.offs.p, sizeof(int64_t) * offs_new.size(), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    L.total = O.total + kept;
    L.off_h.resize((size_t)nc + 1);
    for (int c = 0; c <= nc; ++c) L.off_h[(size_t)c] = O.off_h[(size_t)c] + offs_new[(size_t)c];
    for (int c = 0; c < nc; ++c) L.max_len = std::max(L.max_len, L.off_h[(size_t)c + 1] - L.off_h[(size_t)c]);
    const size_t t1 = (size_t)std::max<int64_t>(L.total, 1);
    TRY(L.off.ensure(sizeof(int64_t) * L.off_h.size(), 0, st, true));
    CK(cudaMemcpyAsync(L.off.p, L.off_h.data(), sizeof(int64_t) * L.off_h.size(), cudaMemcpyHostToDevice, st));
    TRY(L.payload.ensure(t1 * (size_t)rb, 0, st, true));
    TRY(L.rows.ensure(sizeof(int64_t) * t1, 0, st, true));
    TRY(L.labels.ensure(sizeof(int64_t) * t1, 0, st, true));
    const bool has_dead = !O.dead_h.empty();
    if (has_dead) TRY(L.dead.ensure(t1, 0, st, true));
    if (cos_norms) TRY(L.norms.ensure(sizeof(float) * t1, 0, st, true));

    ExtendMergeParams mp{};
    mp.off_old = O.off.as<int64_t>(); mp.offs_new = sc.offs.as<int64_t>(); mp.off_merged = L.off.as<int64_t>();
    mp.order = sc.vals_out.as<int32_t>(); mp.nc = nc;
    auto col = [&](const void* old_src, const void* new_src, DevBuf& dst, int64_t row_bytes, int fold) {
        ExtendMergeColumn& c = mp.col[mp.ncols++];
        c.old_src = (const uint8_t*)old_src; c.new_src = (const uint8_t*)new_src; c.dst = dst.as<uint8_t>();
        c.row_bytes = row_bytes; c.fold_flags = fold;
    };
    col(O.payload.p, pq ? codes.p : (const void*)bd.X, L.payload, rb, 0);
    col(O.rows.p, bd.rows.p, L.rows, 8, 0);
    col(O.labels.p, bd.labels.p, L.labels, 8, 0);
    if (has_dead) col(O.dead.p, nullptr, L.dead, 1, 1);
    if (cos_norms) col(O.norms.p, nnorm.p, L.norms, 4, 0);
    CK(launch_extend_merge(mp, L.total, st));
    CK(cudaStreamSynchronize(st));
    if (has_dead) {
        L.dead_h.assign((size_t)L.total, 0);
        for (int c = 0; c < nc; ++c) {
            const int64_t o = O.off_h[(size_t)c], len = O.off_h[(size_t)c + 1] - o;
            for (int64_t i = 0; i < len; ++i) L.dead_h[(size_t)(o + offs_new[(size_t)c] + i)] = O.dead_h[(size_t)(o + i)] ? 1 : 0;
        }
        L.ndead = O.ndead;  // a flagged entry stays flagged (shadowed becomes deleted), appended entries carry no flag
    }
    S.moved = buffered_rows(h);
    S.noop = false;
    return PYROPE_OK;
}

// A MaxScans budget walks the probed lists entry by entry and never counts a deleted or shadowed entry
// (IvfFlatVectorIndex.cs:209-212), so a budgeted IVF_FLAT search over lists that hold such entries scans a
// compacted VIEW of them (dead entries squeezed out, offsets recomputed).  The lists themselves are left alone:
// a shadowed entry's position still decides where its replacement lands at the next Build (:91-108).
int compact_lists(Index* h) {
    if (h->lists.ndead == 0 || h->bv_version == h->lists_version) return PYROPE_OK;
    cudaStream_t st = h->stream;
    std::vector<int64_t> keep;
    keep.reserve((size_t)h->lists.total);
    std::vector<int64_t> noff((size_t)h->nc + 1, 0);
    for (int c = 0; c < h->nc; ++c) {
        for (int64_t i = h->lists.off_h[(size_t)c]; i < h->lists.off_h[(size_t)c + 1]; ++i)
            if (!h->lists.dead_h[(size_t)i]) keep.push_back(i);
        noff[(size_t)c + 1] = (int64_t)keep.size();
    }
    const int64_t n = (int64_t)keep.size();
    const size_t n1 = (size_t)std::max<int64_t>(n, 1);
    DevBuf idx;
    TRY(idx.ensure(sizeof(int64_t) * n1, 0, st, true));
    CK(cudaMemcpyAsync(idx.p, keep.data(), sizeof(int64_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    TRY(h->bv_vecs.ensure(sizeof(float) * n1 * h->dim, 0, st));
    TRY(h->bv_labels.ensure(sizeof(int64_t) * n1, 0, st));
    TRY(h->bv_off.ensure(sizeof(int64_t) * noff.size(), 0, st));
    CK(launch_gather_rows(h->lists.payload.p, (int64_t)h->dim * 4, idx.as<int64_t>(), n, h->bv_vecs.p, st));
    CK(launch_gather_rows(h->lists.labels.p, 8, idx.as<int64_t>(), n, h->bv_labels.p, st));
    if (h->metric == kCosine) {
        TRY(h->bv_norms.ensure(sizeof(float) * n1, 0, st));
        CK(launch_gather_rows(h->lists.norms.p, 4, idx.as<int64_t>(), n, h->bv_norms.p, st));
    }
    CK(cudaMemcpyAsync(h->bv_off.p, noff.data(), sizeof(int64_t) * noff.size(), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    h->bv_version = h->lists_version;
    return PYROPE_OK;
}

// ------------------------------------------------------------------------------------------
// search
// ------------------------------------------------------------------------------------------
// scan position cut-off so that exactly min(max_scans, live) live rows precede it
int64_t segment_cutoff(const Segment& s, int64_t max_scans) {
    if (max_scans < 0) return s.nslots;
    if (max_scans == 0) return 0;
    if (s.ndead == 0) return std::min<int64_t>(max_scans, s.nslots);
    int64_t seen = 0;
    for (int64_t i = 0; i < s.nslots; ++i) {
        if (!s.dead_h[(size_t)i]) {
            if (++seen == max_scans) return i + 1;
        }
    }
    return s.nslots;
}

// norms (cosine): the exact row norms of X, which decide which rows score 0 (tc_rowterms_kernel)
int ensure_tc_operand(TcOperand& op, const float* X, int64_t n, int dim, int metric, const uint8_t* dead,
                      cudaStream_t st, const float* norms) {
    if (op.dirty) op.rows_valid = 0;
    const size_t keep_e = (size_t)op.rows_valid * dim * sizeof(float), keep_r = (size_t)op.rows_valid * sizeof(float);
    TRY(op.hi.ensure(sizeof(float) * (size_t)n * dim, keep_e, st));
    TRY(op.lo.ensure(sizeof(float) * (size_t)n * dim, keep_e, st));
    TRY(op.scale.ensure(sizeof(float) * (size_t)n, keep_r, st));
    TRY(op.bias.ensure(sizeof(float) * (size_t)n, keep_r, st));
    if (!op.amax.p) {
        TRY(op.amax.ensure(sizeof(float), 0, st, true));
        op.rows_valid = 0;
    }
    if (op.rows_valid == 0) CK(cudaMemsetAsync(op.amax.p, 0, sizeof(float), st));
    if (op.rows_valid < n) {
        CK(launch_tc_prepare(X, n, dim, metric, dead, op.hi.as<float>(), op.lo.as<float>(), op.scale.as<float>(),
                             op.bias.as<float>(), op.rows_valid, st, metric == kCosine ? norms : nullptr));
        CK(launch_tc_amax(X, n, dim, op.scale.as<float>(), op.amax.as<float>(), op.rows_valid, st));
    }
    op.rows_valid = n;
    op.dirty = false;
    return PYROPE_OK;
}

__global__ void fill_empty_kernel(float* s, int64_t* l, int32_t* c, int64_t nq, int k) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nq * k) { s[i] = 0.f; l[i] = -1; }
    if (c && i < nq) c[i] = 0;
}

// ext_probes: probe lists computed elsewhere ([nq][P] list ids in rank order, -1 = none) — the coarse stage is
// skipped.  probes_only_out: run ONLY the coarse stage and write [nq][P] there (multi-GPU: every rank
// ranks centroids for its slice of the batch, the lists are all-gathered, then every rank scans its shard).
int search_device(Index* h, int64_t nq, const float* dQ, int topk, int64_t max_scans, int nprobe, float* d_scores,
                  int64_t* d_rows, int32_t* d_counts, cudaStream_t st, const int64_t* ext_probes = nullptr,
                  int64_t* probes_only_out = nullptr) {
    Workspace& ws = h->ws;
    const int dim = h->dim, k = topk;
    int launches = 0;
    if (h->last_stream && h->last_stream != st) CK(cudaStreamSynchronize(h->last_stream));
    h->last_stream = st;
    if (!h->ev[0]) {
        for (int i = 0; i < 5; ++i) CK(cudaEventCreate(&h->ev[i]));
        for (int i = 0; i < 2; ++i) CK(cudaEventCreate(&h->evk[i]));
        for (int i = 0; i < 2; ++i) CK(cudaEventCreateWithFlags(&h->evf[i], cudaEventDisableTiming));
        CK(cudaStreamCreateWithFlags(&h->aux, cudaStreamNonBlocking));
    }
    h->ev_valid = false;
    h->evk_valid = false;
    h->dom_kernel = "";
    CK(cudaEventRecord(h->ev[0], st));

    auto fill_empty = [&]() -> int {
        int64_t tot = std::max<int64_t>(nq * std::max(k, 1), nq);
        fill_empty_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(d_scores, d_rows, d_counts, nq, std::max(k, 0));
        CK(cudaGetLastError());
        ++launches;
        return PYROPE_OK;
    };

    // ---- plan the parts
    Segment& seg = h->seg;
    const bool ivf = h->kind != PYROPE_FLAT;
    const int64_t seg_scan = (h->kind == PYROPE_IVF_PQ) ? seg.nslots : segment_cutoff(seg, max_scans);
    const bool scan_seg = seg_scan > 0 && seg.live > 0 && !probes_only_out;
    int64_t seg_live_scanned = 0;
    if (scan_seg) seg_live_scanned = (max_scans >= 0 && h->kind != PYROPE_IVF_PQ) ? std::min<int64_t>(max_scans, seg.live) : seg.live;

    int P = 0;  // probes
    bool scan_lists = false;
    if (ivf && h->built && h->nc > 0 && h->lists.total > 0) {
        int np = nprobe >= 0 ? nprobe : (h->kind == PYROPE_IVF_FLAT ? 3 : 1);
        P = std::min(np, h->nc);
        scan_lists = P > 0;
        if (h->kind == PYROPE_IVF_FLAT && max_scans >= 0 && seg_live_scanned >= max_scans) scan_lists = false;
    }
    if (P > kMaxTopK) return fail(PYROPE_ERR_UNSUPPORTED, "nprobe %d exceeds the supported maximum %d", P, kMaxTopK);
    if (probes_only_out && !scan_lists) return fail(PYROPE_ERR_INVALID_STATE, "index has no inverted lists to probe");
    if (!probes_only_out && (k <= 0 || (!scan_seg && !scan_lists))) {
        TRY(fill_empty());
        CK(cudaEventRecord(h->ev[1], st)); CK(cudaEventRecord(h->ev[2], st)); CK(cudaEventRecord(h->ev[3], st));
        h->ev_valid = true;
        h->last_launches = launches;
        return PYROPE_OK;
    }

    int groups = 0;
    if (scan_lists) {
        int64_t want = (2 * (int64_t)g_num_sms + nq - 1) / nq;
        groups = (int)std::max<int64_t>(1, std::min<int64_t>(want, P));
    }
    const bool use_lm = scan_lists && h->kind == PYROPE_IVF_PQ && !h->pq_force_generic && h->pq_lm_mode != 0 &&
                        ivfpq_lm_supported(dim, h->m, h->k, P, k, nq, h->lists.total, h->lists.max_len);
    const bool use_flm = scan_lists && h->kind == PYROPE_IVF_FLAT && h->pq_lm_mode != 0 && nq >= 64 &&
                         ivfflat_lm_supported(dim, h->metric, P, k, nq, h->lists.total, max_scans >= 0);
    if (use_lm || use_flm) groups = 1;
    int max_parts = kMergeMaxCandidates / k;
    if (max_parts < 1) max_parts = 1;
    if (groups > max_parts - (scan_seg ? 1 : 0)) groups = std::max(1, max_parts - (scan_seg ? 1 : 0));
    const bool use_sq8 = scan_seg && h->kind == PYROPE_FLAT && h->sq8;
    const bool use_tc_seg = scan_seg && !use_sq8 && h->tc_mode != 0 && flat_tc_supported(dim, k) &&
                            (h->tc_mode == 1 || seg_scan >= 8192);
    // the fast coarse stage ranks Pc >= P candidate lists; they are re-ranked in the reference's arithmetic
    const int Pc = std::min(h->nc, std::min(P + 8, kMaxTopK));
    // large centroid tables (and dim <= 128): the query-stationary one-TF32 probe with exact ranking of the survivors
    const bool use_ctc = scan_lists && !ext_probes && h->tc_mode != 0 && h->nc >= 2048 && coarse_tc_supported(dim, h->nc, P);
    const bool use_tc_coarse = !use_ctc && scan_lists && !ext_probes && h->tc_mode != 0 && flat_tc_supported(dim, Pc) &&
                               (h->tc_mode == 1 || h->nc >= 2048);
    int seg_splits = 0;
    if (scan_seg) seg_splits = use_tc_seg ? 1 : use_sq8 ? sq8_pick_splits(nq, seg_scan, k, g_num_sms)
                                                        : flat_scan_pick_splits(nq, seg_scan, k, g_num_sms, std::max(1, max_parts - groups));
    const int parts = seg_splits + groups;
    if ((int64_t)parts * k > kMergeMaxCandidates)
        return fail(PYROPE_ERR_UNSUPPORTED, "topK %d too large for %d partial lists", k, parts);

    TRY(ws.pairs_s.ensure(sizeof(float) * (size_t)nq * parts * k, 0, st));
    TRY(ws.pairs_l.ensure(sizeof(int64_t) * (size_t)nq * parts * k, 0, st));
    PairOut out{ws.pairs_s.as<float>(), ws.pairs_l.as<int64_t>(), parts, 0};

    const float* qnorm = nullptr;
    if (h->metric == kCosine) {
        TRY(ws.qnorm.ensure(sizeof(float) * (size_t)nq, 0, st));
        CK(launch_row_norms_exact(dQ, nq, dim, dim, ws.qnorm.as<float>(), st));
        ++launches;
        qnorm = ws.qnorm.as<float>();
    }

    // tf32 hi / lo copies of the queries: made once per search, by the first stage that needs them (the coarse probe on
    // fp16 copies followed by an ADC scan never does)
    bool qsplit_done = false;
    auto need_qsplit = [&]() -> int {
        if (qsplit_done) return PYROPE_OK;
        TRY(ws.qhi.ensure(sizeof(float) * (size_t)nq * dim, 0, st));
        TRY(ws.qlo.ensure(sizeof(float) * (size_t)nq * dim, 0, st));
        CK(launch_tc_prepare(dQ, nq, dim, h->metric, nullptr, ws.qhi.as<float>(), ws.qlo.as<float>(), nullptr, nullptr, 0, st));
        ++launches;
        qsplit_done = true;
        return PYROPE_OK;
    };
    auto run_tc = [&](TcOperand& op, const float* X, int64_t n_rows, int64_t n_scan_rows, const uint8_t* dead,
                      const float* xnorm, const int64_t* labels, int kk, PairOut po) -> int {
        if (op.dirty || op.rows_valid < n_rows) ++launches;
        TRY(need_qsplit());
        TRY(ensure_tc_operand(op, X, n_rows, dim, h->metric, dead, st, xnorm));
        FlatTcParams tp{};
        tp.Q = dQ; tp.Qhi = ws.qhi.as<float>(); tp.Qlo = ws.qlo.as<float>(); tp.nq = nq; tp.dim = dim;
        tp.X = X; tp.Xhi = op.hi.as<float>(); tp.Xlo = op.lo.as<float>(); tp.n_rows = n_rows; tp.n_scan = n_scan_rows;
        tp.scale = op.scale.as<float>(); tp.bias = op.bias.as<float>(); tp.xnorm = xnorm; tp.qnorm = qnorm; tp.labels = labels;
        tp.metric = h->metric; tp.k = kk; tp.kprime = kk + flat_tc_margin(kk); tp.cap = flat_tc_cap(tp.kprime);
        tp.arith = (h->kind == PYROPE_FLAT) ? 1 : 2;  // BruteForceVectorIndex scores with the *Unsafe variants, IVF with L2Squared / DotProduct
        const bool twopass = flat_tc_twopass(dim, n_scan_rows, tp.kprime);
        tp.splits = twopass ? flat_tc_pick_splits_seeded(nq, n_scan_rows, tp.kprime, g_num_sms)
                            : flat_tc_pick_splits(nq, n_scan_rows, tp.kprime, g_num_sms);
        if (twopass) {
            TRY(ws.tcg.ensure(sizeof(float) * flat_tc_gmax_floats(nq, n_scan_rows), 0, st));
            TRY(ws.tct.ensure(sizeof(float) * (2 * (size_t)flat_tc_nq_pad(nq) + 16), 0, st));  // tau | band | overflow flag
            tp.gmax_ws = ws.tcg.as<float>(); tp.tau_ws = ws.tct.as<float>();
            if (!getenv("PYROPE_TC_PASSA_3X")) tp.amax = op.amax.as<float>();
            launches += 3;
        }
        if (!twopass && flat_tc_oneterm(dim, n_scan_rows, tp.kprime)) {
            TRY(ws.tct.ensure(sizeof(float) * (2 * (size_t)flat_tc_nq_pad(nq) + 16), 0, st));  // (unused tau) | band | overflow flag
            tp.tau_ws = ws.tct.as<float>();
            tp.amax = op.amax.as<float>();
            launches += 2;
            // L2 / IP: the pass runs on fp16 copies of both operands when every table value fits the fp16 range
            static const bool no_f16 = getenv("PYROPE_FLAT_TF32") != nullptr;
            if (!no_f16 && h->metric != kCosine && dim % 8 == 0) {
                if (op.h16_rows < n_rows) {
                    // rows appended since the last search are converted on their own (an in-place change invalidates the
                    // operand and starts from row 0); the running maximum covers every row converted so far
                    const int64_t from = op.h16_rows;
                    if (op.h16.ensure(sizeof(uint16_t) * (size_t)n_rows * dim, sizeof(uint16_t) * (size_t)from * dim, st) != PYROPE_OK) {
                        // no room for another half-size copy of the table: the tf32 pass needs none
                        op.h16.release();
                        op.h16_ok = false;
                        op.h16_rows = n_rows;
                        goto half_done;
                    }
                    TRY(op.xabs.ensure(sizeof(float), 0, st, true));
                    if (from == 0) CK(cudaMemsetAsync(op.xabs.p, 0, sizeof(float), st));
                    CK(launch_tc_half(X + (size_t)from * dim, (n_rows - from) * dim, op.h16.as<uint16_t>() + (size_t)from * dim,
                                      op.xabs.as<float>(), st));
                    float xabs = 0.f;
                    CK(cudaMemcpyAsync(&xabs, op.xabs.p, sizeof(float), cudaMemcpyDeviceToHost, st));
                    CK(cudaStreamSynchronize(st));
                    op.h16_ok = xabs <= kTcHalfMaxAbs;
                    op.h16_rows = n_rows;
                    ++launches;
                }
            half_done:
                if (op.h16_ok && op.h16.p) {
                    TRY(ws.q16.ensure(sizeof(uint16_t) * (size_t)nq * dim, 0, st));
                    TRY(ws.qbad.ensure((size_t)nq, 0, st));
                    CK(launch_tc_half_rows(dQ, nq, dim, ws.q16.p, ws.qbad.as<uint8_t>(), st));
                    ++launches;
                    tp.Q16 = ws.q16.p; tp.X16 = op.h16.p; tp.qbad = ws.qbad.as<uint8_t>();
                }
            }
        }
        const int64_t nq_pad = flat_tc_nq_pad(nq);
        const size_t tparts = (size_t)tp.splits * flat_tc_parts_per_split(tp);
        TRY(ws.tcq.ensure(sizeof(uint64_t) * tparts * nq_pad * tp.cap, 0, st));
        TRY(ws.tcc.ensure(sizeof(int32_t) * tparts * nq_pad, 0, st));
        tp.queue = ws.tcq.as<uint64_t>(); tp.counts = ws.tcc.as<int32_t>(); tp.out = po;
        if (&op == &h->tc_seg && h->kind == PYROPE_FLAT) {
            tp.ev_k0 = h->evk[0]; tp.ev_k1 = h->evk[1];
            h->evk_valid = true;
            // one TF32 term + rigorous band (tau_ws without the two-pass maxima), or the three-term split
            h->dom_kernel = (tp.tau_ws && !tp.gmax_ws) ? (tp.X16 ? "flat_tc_kernel (1xFP16 + band)" : "flat_tc_kernel (1xTF32 + band)")
                                                       : "flat_tc_kernel (3xTF32)";
        }
        CK(launch_flat_tc(tp, st));
        launches += 2;
        return PYROPE_OK;
    };

    // ---- coarse probe: exact FLAT top-P over the centroids
    const int64_t* probes_dev = ext_probes;
    if (scan_lists && !ext_probes) {
        TRY(ws.probes.ensure(sizeof(int64_t) * (size_t)nq * P, 0, st));
        probes_dev = ws.probes.as<int64_t>();
    }
    if (ext_probes) {
        // supplied by the caller
    } else if (use_ctc) {
        TcOperand& op = h->tc_cent;
        if (op.dirty || op.rows_valid < h->nc) ++launches;
        if (op.dirty || op.rows_valid < h->nc) op.h16_rows = 0;
        TRY(ensure_tc_operand(op, h->centroids.as<float>(), h->nc, dim, h->metric, nullptr, st, h->cnorms.as<float>()));
        TRY(ws.ctc.ensure(coarse_tc_scratch_bytes(nq, h->nc, g_num_sms), 0, st));
        CoarseTcParams cp{};
        // L2 / IP, rows a multiple of 16 bytes in fp16: the tensor passes run on fp16 copies (twice the MMA rate, half the
        // operand bytes, the same 10-bit mantissa)
        static const bool no_f16 = getenv("PYROPE_COARSE_TF32") != nullptr;
        if (!no_f16 && h->metric != kCosine && dim % 8 == 0) {
            if (op.h16_rows != h->nc) {
                TRY(op.h16.ensure(sizeof(uint16_t) * (size_t)h->nc * dim, 0, st));
                TRY(op.xabs.ensure(sizeof(float), 0, st, true));
                CK(cudaMemsetAsync(op.xabs.p, 0, sizeof(float), st));
                CK(launch_tc_half(h->centroids.as<float>(), (int64_t)h->nc * dim, op.h16.p, op.xabs.as<float>(), st));
                float xabs = 0.f;
                CK(cudaMemcpyAsync(&xabs, op.xabs.p, sizeof(float), cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
                op.h16_ok = xabs <= kTcHalfMaxAbs;
                op.h16_rows = h->nc;
                ++launches;
            }
            if (op.h16_ok) {
                TRY(ws.q16.ensure(sizeof(uint16_t) * (size_t)nq * dim, 0, st));
                TRY(ws.qbad.ensure((size_t)nq, 0, st));
                CK(launch_tc_half_rows(dQ, nq, dim, ws.q16.p, ws.qbad.as<uint8_t>(), st));
                ++launches;
                cp.Q16 = ws.q16.p; cp.C16 = op.h16.p; cp.qbad = ws.qbad.as<uint8_t>();
            }
        }
        if (!cp.Q16) TRY(need_qsplit());
        cp.Q = dQ; cp.Qhi = ws.qhi.as<float>(); cp.nq = nq; cp.dim = dim; cp.metric = h->metric;
        cp.C = h->centroids.as<float>(); cp.Chi = op.hi.as<float>(); cp.cnorms = h->cnorms.as<float>(); cp.nc = h->nc;
        cp.scale = op.scale.as<float>(); cp.bias = op.bias.as<float>(); cp.amax = op.amax.as<float>();
        cp.nprobe = P; cp.probes_out = ws.probes.as<int64_t>(); cp.scratch = ws.ctc.p; cp.num_sms = g_num_sms;
        CK(launch_coarse_tc(cp, st));
        launches += coarse_tc_launches();
    } else if (scan_lists) {
        TRY(ws.probes_raw.ensure(sizeof(int64_t) * (size_t)nq * Pc, 0, st));
        TRY(ws.probe_scores.ensure(sizeof(float) * (size_t)nq * Pc, 0, st));
        if (use_tc_coarse) {
            TRY(run_tc(h->tc_cent, h->centroids.as<float>(), h->nc, h->nc, nullptr, h->cnorms.as<float>(), nullptr, Pc,
                       PairOut{ws.probe_scores.as<float>(), ws.probes_raw.as<int64_t>(), 1, 0}));
        } else {
            int csplits = flat_scan_pick_splits(nq, h->nc, Pc, g_num_sms, 0);
            int ccap = flat_scan_cap(Pc);
            TRY(ws.queue.ensure(sizeof(uint64_t) * (size_t)csplits * nq * ccap, 0, st));
            TRY(ws.cpairs_s.ensure(sizeof(float) * (size_t)nq * csplits * Pc, 0, st));
            TRY(ws.cpairs_l.ensure(sizeof(int64_t) * (size_t)nq * csplits * Pc, 0, st));
            FlatScanParams cp{};
            cp.Q = dQ; cp.nq = nq; cp.dim = dim; cp.X = h->centroids.as<float>(); cp.n_scan = h->nc;
            cp.dead = nullptr; cp.xnorm = h->cnorms.as<float>(); cp.qnorm = qnorm; cp.labels = nullptr;
            cp.metric = h->metric; cp.k = Pc; cp.splits = csplits; cp.queue = ws.queue.as<uint64_t>(); cp.cap = ccap;
            cp.out = PairOut{ws.cpairs_s.as<float>(), ws.cpairs_l.as<int64_t>(), csplits, 0};
            CK(launch_flat_scan(cp, st));
            CK(launch_merge_pairs(nq, csplits, Pc, Pc, ws.cpairs_s.as<float>(), ws.cpairs_l.as<int64_t>(), Pc, (int64_t)csplits * Pc,
                                  ws.probe_scores.as<float>(), ws.probes_raw.as<int64_t>(), nullptr, st));
            launches += 2;
        }
        // IvfFlatVectorIndex.cs:186-198 / IvfPqVectorIndex.cs:141-150: rank by the reference's own arithmetic
        CK(launch_coarse_rerank_exact(h->metric, dim, nq, dQ, h->centroids.as<float>(), h->cnorms.as<float>(), h->nc,
                                      ws.probes_raw.as<int64_t>(), ws.probe_scores.as<float>(), Pc, ws.probes.as<int64_t>(),
                                      nullptr, P, (h->kind == PYROPE_IVF_FLAT && max_scans >= 0) ? 1 : 0, st));
        ++launches;
    }
    CK(cudaEventRecord(h->ev[1], st));
    if (probes_only_out) {
        CK(cudaMemcpyAsync(probes_only_out, probes_dev, sizeof(int64_t) * (size_t)nq * P, cudaMemcpyDeviceToDevice, st));
        CK(cudaEventRecord(h->ev[2], st)); CK(cudaEventRecord(h->ev[3], st));
        h->ev_valid = true;
        h->last_launches = launches;
        return PYROPE_OK;
    }

    bool direct_out = false;
    // ---- buffer / base scan
    if (scan_seg && use_tc_seg) {
        PairOut po = out;
        po.part_base = 0;
        if (seg.tc_dirty) { h->tc_seg.invalidate(); seg.tc_dirty = false; }
        TRY(run_tc(h->tc_seg, seg.X.as<float>(), seg.nslots, seg_scan, seg.ndead > 0 ? seg.dead.as<uint8_t>() : nullptr,
                   seg.norms.as<float>(), seg.labels.as<int64_t>(), k, po));
    } else if (use_sq8) {
        // quantised branch of BruteForceVectorIndex.Search (:297-336): the query gets its own min / max, rows are
        // ranked by the integer distance between the byte vectors
        TRY(ws.q8.ensure((size_t)nq * h->dpad, 0, st));
        CK(launch_sq8_quantize(dQ, nq, dim, dim, ws.q8.as<uint8_t>(), h->dpad, nullptr, st));
        PairOut po = out;
        po.part_base = 0;
        CK(launch_sq8_scan(ws.q8.as<uint8_t>(), nq, h->dpad, h->x8.as<uint8_t>(), seg_scan,
                           seg.ndead > 0 ? seg.dead.as<uint8_t>() : nullptr, h->qvalid8.as<uint8_t>(), seg.labels.as<int64_t>(),
                           h->metric, k, seg_splits, po, st));
        launches += 2;
        h->dom_kernel = "sq8_scan_kernel";
    } else if (scan_seg) {
        int cap = flat_scan_cap(k);
        TRY(ws.queue.ensure(sizeof(uint64_t) * (size_t)seg_splits * nq * cap, 0, st));
        FlatScanParams fp{};
        fp.Q = dQ; fp.nq = nq; fp.dim = dim; fp.X = seg.X.as<float>(); fp.n_scan = seg_scan;
        fp.dead = seg.ndead > 0 ? seg.dead.as<uint8_t>() : nullptr;
        fp.xnorm = seg.norms.as<float>(); fp.qnorm = qnorm; fp.labels = seg.labels.as<int64_t>();
        fp.metric = h->metric; fp.k = k; fp.splits = seg_splits; fp.queue = ws.queue.as<uint64_t>(); fp.cap = cap;
        fp.out = out; fp.out.part_base = 0;
        CK(launch_flat_scan(fp, st));
        ++launches;
    }
    // ---- list scan
    if (scan_lists) {
        const uint8_t* ldead = h->lists.ndead > 0 ? h->lists.dead.as<uint8_t>() : nullptr;
        if (h->kind == PYROPE_IVF_FLAT) {
            const int32_t* allow = nullptr;
            const bool budget_view = max_scans >= 0 && h->lists.ndead > 0;
            if (budget_view && h->bv_version != h->lists_version)
                return fail(PYROPE_ERR_INVALID_STATE, "budgeted IVF_FLAT search without a compacted list view");
            if (max_scans >= 0) {
                TRY(ws.allow.ensure(sizeof(int32_t) * (size_t)nq * P, 0, st));
                CK(launch_probe_allow(probes_dev, nq, P, (budget_view ? h->bv_off : h->lists.off).as<int64_t>(),
                                      max_scans - seg_live_scanned, ws.allow.as<int32_t>(), st));
                ++launches;
                allow = ws.allow.as<int32_t>();
            }
            IvfFlatScanParams ip{};
            ip.Q = dQ; ip.nq = nq; ip.dim = dim; ip.probes = probes_dev; ip.nprobe = P; ip.allow = allow;
            ip.list_off = h->lists.off.as<int64_t>(); ip.vecs = h->lists.payload.as<float>(); ip.dead = ldead;
            ip.norms = h->lists.norms.as<float>(); ip.labels = h->lists.labels.as<int64_t>(); ip.qnorm = qnorm;
            if (budget_view) {
                ip.list_off = h->bv_off.as<int64_t>(); ip.vecs = h->bv_vecs.as<float>(); ip.dead = nullptr;
                ip.norms = h->bv_norms.as<float>(); ip.labels = h->bv_labels.as<int64_t>();
            }
            ip.metric = h->metric; ip.k = k; ip.groups = groups;
            ip.out = out; ip.out.part_base = seg_splits;
            if (use_flm) {
                TRY(ws.lm.ensure(ivfflat_lm_scratch_bytes(nq, P, k, h->nc), 0, st));
                ip.ev_k0 = h->evk[0]; ip.ev_k1 = h->evk[1];
                h->evk_valid = true;
                h->dom_kernel = "ivf_lm_scan_kernel";
                CK(launch_ivfflat_scan_lm(ip, h->nc, ws.lm.p, g_num_sms, st));
                h->lm_nq = nq; h->lm_P = P; h->lm_k = k;
                launches += ivfflat_lm_launches() - 1;
            } else {
                CK(launch_ivfflat_scan(ip, st));
            }
        } else {
            IvfPqScanParams pp{};
            pp.Q = dQ; pp.nq = nq; pp.dim = dim; pp.probes = probes_dev; pp.nprobe = P;
            pp.list_off = h->lists.off.as<int64_t>(); pp.nlist = h->nc; pp.centroids = h->centroids.as<float>();
            pp.codebook = h->codebook.as<float>(); pp.m = h->m; pp.ksub = h->k;
            pp.codes = h->lists.payload.as<uint8_t>(); pp.dead = ldead; pp.labels = h->lists.labels.as<int64_t>();
            pp.k = k; pp.groups = groups; pp.force_generic = h->pq_force_generic;
            pp.out = out; pp.out.part_base = seg_splits;
            if (use_lm && parts == 1) {  // the only part: the final kernel writes the search's output itself, no merge pass
                pp.out = PairOut{d_scores, d_rows, 1, 0};
                pp.out_counts = d_counts;
                direct_out = true;
            }
            if (use_lm && !h->peer_thr.empty() && nq <= h->thr_cap) {
                // bounds the peers prove for this batch land in thr_pub while the scan runs.  Every word carries the
                // batch epoch, so nothing is cleared and a peer that is a batch behind (or ahead) cannot disturb this one
                if (!h->thr_epoch_set) h->thr_epoch = h->thr_epoch + 1 == 0 ? 1 : h->thr_epoch + 1;
                h->thr_epoch_set = false;
                pp.epoch = h->thr_epoch;
                pp.thr_pub = h->thr_pub.as<unsigned long long>();
                pp.n_peers = (int)h->peer_thr.size();
                for (int r = 0; r < pp.n_peers; ++r) pp.peer_thr[r] = h->peer_thr[(size_t)r];
            }
            if (use_lm) {
                if (h->m != 16) {  // the scan's 16-table view of this quantiser
                    if (!h->lm_cb16_ok) {
                        TRY(h->lm_cb16.ensure(sizeof(float) * (size_t)h->k * dim, 0, st, true));
                        CK(launch_pq_lm_expand_codebook(h->codebook.as<float>(), h->m, h->k, dim, h->lm_cb16.as<float>(), st));
                        h->lm_cb16_ok = true;
                        h->pq_cmax_ok = false;
                        ++launches;
                    }
                    if (!h->lm_codes16_ok) {
                        TRY(h->lm_codes16.ensure((size_t)std::max<int64_t>(h->lists.total, 1) * 16, 0, st, true));
                        CK(launch_pq_lm_expand_codes(h->lists.payload.as<uint8_t>(), h->lists.total, h->m, h->lm_codes16.as<uint8_t>(), st));
                        h->lm_codes16_ok = true;
                        ++launches;
                    }
                    pp.lm_codebook = h->lm_cb16.as<float>();
                    pp.lm_codes = h->lm_codes16.as<uint8_t>();
                }
                if (!h->pq_cmax_ok) {  // once per codebook
                    TRY(h->pq_cmax.ensure(sizeof(float) * 16, 0, st, true));
                    CK(launch_pq_cmax(pp.lm_codebook ? pp.lm_codebook : h->codebook.as<float>(), h->k, dim / 16, h->pq_cmax.as<float>(), st));
                    h->pq_cmax_ok = true;
                    ++launches;
                }
                pp.cmax = h->pq_cmax.as<float>();
                TRY(ws.lm.ensure(ivfpq_lm_scratch_bytes(nq, P, k, h->nc, dim, h->lists.max_len), 0, st));
                pp.max_list_len = h->lists.max_len;
                pp.ev_k0 = h->evk[0]; pp.ev_k1 = h->evk[1];
                pp.aux_stream = h->aux; pp.ev_fork = h->evf[0]; pp.ev_join = h->evf[1];
                h->evk_valid = true;
                h->dom_kernel = "ivfpq_lm_scan_kernel";
                CK(launch_ivfpq_scan_lm(pp, ws.lm.p, g_num_sms, st));
                h->lm_nq = nq; h->lm_P = P; h->lm_k = k;
                launches += ivfpq_lm_launches() - 1;
            } else {
                CK(launch_ivfpq_scan(pp, st));
            }
        }
        ++launches;
    }
    CK(cudaEventRecord(h->ev[2], st));
    if (!direct_out) {
        CK(launch_merge_pairs(nq, parts, k, k, out.scores, out.labels, k, (int64_t)parts * k, d_scores, d_rows, d_counts, st));
        ++launches;
    }
    CK(cudaEventRecord(h->ev[3], st));
    h->ev_valid = true;
    h->last_launches = launches;
    return PYROPE_OK;
}

int validate_search(Index* h, int64_t nq, const float* Q, int topk) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (nq < 0 || (nq > 0 && !Q)) return fail(PYROPE_ERR_INVALID_ARG, "query is null");
    if (h->kind == PYROPE_FLAT && topk <= 0) return fail(PYROPE_ERR_OUT_OF_RANGE, "topK must be positive.");
    if (topk > kMaxTopK) return fail(PYROPE_ERR_UNSUPPORTED, "topK %d exceeds the supported maximum %d", topk, kMaxTopK);
    return PYROPE_OK;
}

}  // namespace

// ==============================================================================================
// C ABI
// ==============================================================================================
extern "C" {

const char* pyrope_last_error(void) { return g_err.c_str(); }
// kept for shims that bind the per-module readers: every module reports through the one channel
const char* pyrope_sharded_last_error(void) { return g_err.c_str(); }
const char* pyrope_peer_last_error(void) { return g_err.c_str(); }
const char* pyrope_batcher_last_error(void) { return g_err.c_str(); }
const char* pyrope_vindex_last_error(void) { return g_err.c_str(); }
const char* pyrope_formats_last_error(void) { return g_err.c_str(); }
int pyrope_version(void) { return 100; }

int pyrope_gpu_device_count(int* out) {
    if (!out) return fail(PYROPE_ERR_INVALID_ARG, "out is null");
    CK(cudaGetDeviceCount(out));
    return PYROPE_OK;
}

int pyrope_gpu_init(int device) {
    if (device >= 0) CK(cudaSetDevice(device));
    CK(cudaFree(0));
    g_inited = false;
    return ensure_init();
}

int pyrope_gpu_shutdown(void) {
    g_inited = false;
    return PYROPE_OK;
}

int pyrope_index_create(int kind, int dim, int metric, int nlist, int pq_m, int pq_k, pyrope_index** out) {
    if (!out) return fail(PYROPE_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    if (kind < PYROPE_FLAT || kind > PYROPE_IVF_PQ) return fail(PYROPE_ERR_INVALID_ARG, "unknown index kind %d", kind);
    if (metric < PYROPE_L2 || metric > PYROPE_COSINE) return fail(PYROPE_ERR_INVALID_ARG, "unknown metric %d", metric);
    if (dim <= 0) return fail(PYROPE_ERR_OUT_OF_RANGE, "Dimension must be positive.");
    if (kind == PYROPE_IVF_PQ) {
        if (pq_m <= 0 || dim % pq_m != 0) return fail(PYROPE_ERR_INVALID_ARG, "Dimension must be divisible by M");
        if (pq_k > 256) return fail(PYROPE_ERR_INVALID_ARG, "K must be <= 256 for byte encoding");
        if (pq_k <= 0) return fail(PYROPE_ERR_INVALID_ARG, "K must be positive");
    }
    TRY(ensure_init());
    Index* h = new (std::nothrow) Index();
    if (!h) return fail(PYROPE_ERR_OOM, "out of host memory");
    h->kind = kind; h->dim = dim; h->metric = metric; h->nlist = nlist;
    if (kind == PYROPE_IVF_PQ) { h->m = pq_m; h->k = pq_k; h->sub = dim / pq_m; }
    h->seg.dim = dim;
    h->seg.cosine = (metric == PYROPE_COSINE);
    h->seg.reuse_slots = (kind != PYROPE_FLAT);
    cudaGetDevice(&h->device);
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete h;
        return fail(PYROPE_ERR_CUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(e));
    }
    const char* g = getenv("PYROPE_PQ_GENERIC");
    h->pq_force_generic = (g && g[0] == '1') ? 1 : 0;
    const char* lmv = getenv("PYROPE_PQ_LM");
    h->pq_lm_mode = (lmv && lmv[0] == '0') ? 0 : -1;
    const char* t = getenv("PYROPE_FLAT_TC");
    h->tc_mode = (t && t[0] == '0') ? 0 : (t && t[0] == '1') ? 1 : -1;
    *out = h;
    return PYROPE_OK;
}

int pyrope_index_destroy(pyrope_index* h) {
    if (!h) return PYROPE_OK;
    cudaStreamSynchronize(h->stream);
    for (unsigned long long* pp : h->peer_thr) if (h->peer_ipc) cudaIpcCloseMemHandle(pp);
    h->peer_thr.clear();
    if (h->last_stream) cudaStreamSynchronize(h->last_stream);
    for (int i = 0; i < 5; ++i)
        if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    for (int i = 0; i < 2; ++i)
        if (h->evk[i]) cudaEventDestroy(h->evk[i]);
    for (int i = 0; i < 2; ++i)
        if (h->evf[i]) cudaEventDestroy(h->evf[i]);
    if (h->aux) { cudaStreamSynchronize(h->aux); cudaStreamDestroy(h->aux); }
    cudaStreamDestroy(h->stream);
    delete h;
    return PYROPE_OK;
}

int pyrope_index_reserve(pyrope_index* h, int64_t n_rows) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::lock_guard<std::mutex> g(h->mu);
    TRY(h->seg.reserve(n_rows, h->stream, true));
    CK(cudaStreamSynchronize(h->stream));
    return PYROPE_OK;
}

int pyrope_index_add_batch(pyrope_index* h, int64_t n, const float* X, const int64_t* labels, int64_t* first_row_out) {
    return add_common(h, n, X, false, labels, first_row_out);
}
int pyrope_index_add_batch_device(pyrope_index* h, int64_t n, const float* dX, const int64_t* d_labels,
                                  int64_t* first_row_out) {
    return add_common(h, n, dX, true, d_labels, first_row_out);
}

int pyrope_index_update_row(pyrope_index* h, int64_t row, const float* x) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (!x) return fail(PYROPE_ERR_INVALID_ARG, "vector is null");
    std::lock_guard<std::mutex> g(h->mu);
    TRY(wait_last_search(h));
    Segment& s = h->seg;
    int64_t slot;
    if (h->kind == PYROPE_FLAT) {
        if (row < 0 || row >= s.nslots) return fail(PYROPE_ERR_NOT_FOUND, "row %lld does not exist", (long long)row);
        slot = row;
    } else {
        if (row < 0 || row >= h->next_row) return fail(PYROPE_ERR_NOT_FOUND, "row %lld does not exist", (long long)row);
        TRY(rebuild_row_loc(h));
        slot = h->row_loc[(size_t)row];
        if (slot < 0) return fail(PYROPE_ERR_NOT_FOUND, "row %lld is not in the write buffer", (long long)row);
    }
    cudaStream_t st = h->stream;
    CK(cudaMemcpyAsync(s.X.as<float>() + slot * s.dim, x, sizeof(float) * s.dim, cudaMemcpyHostToDevice, st));
    if (s.cosine) CK(launch_row_norms_exact(s.X.as<float>() + slot * s.dim, 1, s.dim, s.dim, s.norms.as<float>() + slot, st));
    s.tc_dirty = true;
    if (h->kind == PYROPE_FLAT) TRY(sq8_rows(h, slot, 1));  // :209-214: quantised form refreshed, or reset to empty
    if (s.dead_h[(size_t)slot]) {  // FLAT Upsert un-deletes (BruteForceVectorIndex.cs:200-203)
        CK(cudaMemsetAsync(s.dead.as<uint8_t>() + slot, 0, 1, st));
        s.dead_h[(size_t)slot] = 0;
        s.ndead--;
        s.live++;
    }
    CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

int pyrope_index_delete_row(pyrope_index* h, int64_t row) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::lock_guard<std::mutex> g(h->mu);
    TRY(wait_last_search(h));
    Segment& s = h->seg;
    cudaStream_t st = h->stream;
    if (h->kind == PYROPE_FLAT) {
        if (row < 0 || row >= s.nslots || s.dead_h[(size_t)row]) return fail(PYROPE_ERR_NOT_FOUND, "row %lld not found", (long long)row);
        CK(cudaMemsetAsync(s.dead.as<uint8_t>() + row, 1, 1, st));
        s.tc_dirty = true;
        s.dead_h[(size_t)row] = 1;
        s.ndead++;
        s.live--;
        CK(cudaStreamSynchronize(st));
        return PYROPE_OK;
    }
    if (row < 0 || row >= h->next_row) return fail(PYROPE_ERR_NOT_FOUND, "row %lld not found", (long long)row);
    TRY(rebuild_row_loc(h));
    int64_t loc = h->row_loc[(size_t)row];
    if (loc == -1) return fail(PYROPE_ERR_NOT_FOUND, "row %lld not found", (long long)row);
    if (loc >= 0) {
        CK(cudaMemsetAsync(s.dead.as<uint8_t>() + loc, 1, 1, st));
        s.tc_dirty = true;
        s.dead_h[(size_t)loc] = 1;
        s.slot_row[(size_t)loc] = -1;
        s.ndead++;
        s.live--;
        s.free_stack.push_back(loc);
        h->row_loc[(size_t)row] = -1;
    } else {
        if (h->kind == PYROPE_IVF_PQ)  // IvfPqVectorIndex.cs:48-53: Delete only touches the buffer
            return fail(PYROPE_ERR_NOT_FOUND, "row %lld is encoded in a list; IVF_PQ deletes only buffered rows", (long long)row);
        TRY(set_list_flag(h, {-2 - loc}, 1, true));
        h->row_loc[(size_t)row] = -1;
    }
    CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

int pyrope_index_shadow_row(pyrope_index* h, int64_t row, int shadowed) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::lock_guard<std::mutex> g(h->mu);
    TRY(wait_last_search(h));
    if (h->kind == PYROPE_FLAT) return fail(PYROPE_ERR_INVALID_STATE, "FLAT rows cannot be shadowed");
    if (row < 0 || row >= h->next_row) return fail(PYROPE_ERR_NOT_FOUND, "row %lld not found", (long long)row);
    TRY(rebuild_row_loc(h));
    int64_t loc = h->row_loc[(size_t)row];
    if (loc > -2) return fail(PYROPE_ERR_NOT_FOUND, "row %lld is not in an inverted list", (long long)row);
    TRY(set_list_flag(h, {-2 - loc}, 2, shadowed != 0));
    CK(cudaStreamSynchronize(h->stream));
    return PYROPE_OK;
}

int pyrope_index_set_labels(pyrope_index* h, int64_t n_rows, const int64_t* labels_by_row) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (n_rows < h->next_row || (n_rows > 0 && !labels_by_row))
        return fail(PYROPE_ERR_INVALID_ARG, "labels for %lld rows needed, %lld given", (long long)h->next_row, (long long)n_rows);
    std::lock_guard<std::mutex> g(h->mu);
    TRY(wait_last_search(h));
    cudaStream_t st = h->stream;
    Segment& s = h->seg;
    if (s.nslots > 0) {
        std::vector<int64_t> L((size_t)s.nslots);
        for (int64_t i = 0; i < s.nslots; ++i) {
            const int64_t row = h->kind == PYROPE_FLAT ? i : s.slot_row[(size_t)i];
            L[(size_t)i] = row >= 0 ? labels_by_row[(size_t)row] : -1;
        }
        CK(cudaMemcpyAsync(s.labels.p, L.data(), sizeof(int64_t) * L.size(), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
    }
    if (h->kind != PYROPE_FLAT && h->lists.total > 0) {
        DevBuf dl;
        TRY(dl.ensure(sizeof(int64_t) * (size_t)n_rows, 0, st, true));
        CK(cudaMemcpyAsync(dl.p, labels_by_row, sizeof(int64_t) * (size_t)n_rows, cudaMemcpyHostToDevice, st));
        CK(launch_gather_rows(dl.p, 8, h->lists.rows.as<int64_t>(), h->lists.total, h->lists.labels.p, st));
        CK(cudaStreamSynchronize(st));
    }
    return PYROPE_OK;
}

int pyrope_index_set_quantization(pyrope_index* h, int enable) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (h->kind != PYROPE_FLAT) return fail(PYROPE_ERR_INVALID_STATE, "only the FLAT index has a quantised scan");
    std::lock_guard<std::mutex> g(h->mu);
    TRY(wait_last_search(h));
    h->sq8 = enable != 0;
    if (h->sq8 && !h->x8.p) {  // first use: rows that exist already have no quantised form (added while the flag was off)
        h->dpad = (h->dim + 15) / 16 * 16;
        const int64_t cap = std::max<int64_t>(h->seg.cap, 1);
        TRY(h->x8.ensure((size_t)cap * h->dpad, 0, h->stream, true));
        TRY(h->qvalid8.ensure((size_t)cap, 0, h->stream, true));
        CK(cudaMemsetAsync(h->qvalid8.p, 0, h->qvalid8.bytes, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        h->x8_cap = cap;
    }
    return PYROPE_OK;
}

int pyrope_index_build(pyrope_index* h) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::lock_guard<std::mutex> g(h->mu);
    Staged S(*h);
    TRY(build_prepare(*h, S));
    install(h, S);
    return PYROPE_OK;
}

int pyrope_index_extend(pyrope_index* h) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::lock_guard<std::mutex> g(h->mu);
    Staged S(*h);
    TRY(extend_prepare(*h, S));
    install(h, S);
    return PYROPE_OK;
}

int pyrope_index_set_train_params(pyrope_index* h, int64_t max_train_rows, int max_iter) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    h->max_train_rows = max_train_rows;
    h->max_iter = max_iter;
    return PYROPE_OK;
}

int pyrope_index_set_codebooks(pyrope_index* h, int n_centroids, const float* centroids, const float* pq_codebooks) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (h->kind == PYROPE_FLAT) return fail(PYROPE_ERR_INVALID_STATE, "FLAT has no codebooks");
    if (n_centroids <= 0 || !centroids) return fail(PYROPE_ERR_INVALID_ARG, "centroids missing");
    if (h->kind == PYROPE_IVF_PQ && !pq_codebooks) return fail(PYROPE_ERR_INVALID_ARG, "pq codebooks missing");
    std::lock_guard<std::mutex> g(h->mu);
    cudaStream_t st = h->stream;
    TRY(h->centroids.ensure(sizeof(float) * (size_t)n_centroids * h->dim, 0, st, true));
    CK(cudaMemcpyAsync(h->centroids.p, centroids, sizeof(float) * (size_t)n_centroids * h->dim, cudaMemcpyDefault, st));
    if (h->kind == PYROPE_IVF_PQ) {
        size_t cb = sizeof(float) * (size_t)h->m * h->k * h->sub;
        TRY(h->codebook.ensure(cb, 0, st, true));
        CK(cudaMemcpyAsync(h->codebook.p, pq_codebooks, cb, cudaMemcpyDefault, st));
        h->pq_cmax_ok = false; h->lm_cb16_ok = false;
        h->ksub.assign((size_t)h->m, h->k);
    }
    CK(cudaStreamSynchronize(st));
    h->nc = n_centroids;
    h->frozen = true;
    h->tc_cent.invalidate();
    return PYROPE_OK;
}

int pyrope_index_set_shard(pyrope_index* h, int rank, int world) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (h->kind == PYROPE_FLAT) return fail(PYROPE_ERR_INVALID_STATE, "FLAT shards by rows: add only this rank's rows");
    if (world < 1 || rank < 0 || rank >= world) return fail(PYROPE_ERR_INVALID_ARG, "bad shard %d/%d", rank, world);
    h->shard_rank = rank;
    h->shard_world = world;
    return PYROPE_OK;
}

}  // extern "C"
namespace {
// this rank's published-threshold array: (re)allocated zeroed for batches of up to max_queries queries
int thr_array_ensure(Index* h, int64_t max_queries) {
    if (h->kind != PYROPE_IVF_PQ) return fail(PYROPE_ERR_INVALID_STATE, "threshold exchange exists on the IVF_PQ list-major path only");
    if (max_queries <= h->thr_cap && h->thr_pub.p) return PYROPE_OK;
    if (!h->peer_thr.empty()) return fail(PYROPE_ERR_INVALID_STATE, "peers are already attached");
    CK(cudaStreamSynchronize(h->stream));
    if (h->last_stream) CK(cudaStreamSynchronize(h->last_stream));
    h->thr_pub.release();
    TRY(h->thr_pub.ensure(sizeof(unsigned long long) * (size_t)max_queries, 0, h->stream, true));
    CK(cudaMemsetAsync(h->thr_pub.p, 0, h->thr_pub.bytes, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->thr_cap = max_queries;
    return PYROPE_OK;
}
}  // namespace
extern "C" {

int pyrope_index_threshold_exchange_handle(pyrope_index* h, int64_t max_queries, void* handle_out) {
    if (!h || !handle_out || max_queries <= 0) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    std::lock_guard<std::mutex> g(h->mu);
    if (!h->peer_thr.empty()) return fail(PYROPE_ERR_INVALID_STATE, "peers are already attached");
    TRY(thr_array_ensure(h, max_queries));
    cudaIpcMemHandle_t hd;
    CK(cudaIpcGetMemHandle(&hd, h->thr_pub.p));
    memcpy(handle_out, &hd, sizeof hd);
    return PYROPE_OK;
}

int pyrope_index_threshold_exchange_array(pyrope_index* h, int64_t max_queries, void** d_array_out) {
    if (!h || !d_array_out || max_queries <= 0) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    std::lock_guard<std::mutex> g(h->mu);
    TRY(thr_array_ensure(h, max_queries));
    *d_array_out = h->thr_pub.p;
    return PYROPE_OK;
}

int pyrope_index_threshold_exchange_attach(pyrope_index* h, int world, int rank, void* const* arrays) {
    if (!h || !arrays) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    if (world < 2 || world > 8 || rank < 0 || rank >= world) return fail(PYROPE_ERR_INVALID_ARG, "world must be 2..8");
    std::lock_guard<std::mutex> g(h->mu);
    if (!h->thr_pub.p) return fail(PYROPE_ERR_INVALID_STATE, "call pyrope_index_threshold_exchange_array first");
    if (!h->peer_thr.empty()) return fail(PYROPE_ERR_INVALID_STATE, "peers are already attached");
    for (int r = 0; r < world; ++r) {
        if (r == rank) continue;
        if (!arrays[r]) { h->peer_thr.clear(); return fail(PYROPE_ERR_INVALID_ARG, "array of shard %d is null", r); }
        h->peer_thr.push_back(reinterpret_cast<unsigned long long*>(arrays[r]));
    }
    h->peer_ipc = false;  // same-process device pointers (peer access enabled by the caller): nothing to close
    return PYROPE_OK;
}

int pyrope_index_threshold_exchange_open(pyrope_index* h, int world, int rank, const void* handles) {
    if (!h || !handles) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    if (world < 2 || world > 8 || rank < 0 || rank >= world) return fail(PYROPE_ERR_INVALID_ARG, "world must be 2..8");
    std::lock_guard<std::mutex> g(h->mu);
    if (!h->thr_pub.p) return fail(PYROPE_ERR_INVALID_STATE, "call pyrope_index_threshold_exchange_handle first");
    for (int r = 0; r < world; ++r) {
        if (r == rank) continue;
        cudaIpcMemHandle_t hd;
        memcpy(&hd, (const char*)handles + (size_t)r * sizeof hd, sizeof hd);
        void* pp = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&pp, hd, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            for (unsigned long long* q : h->peer_thr) cudaIpcCloseMemHandle(q);
            h->peer_thr.clear();
            return fail(PYROPE_ERR_CUDA, "cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
        }
        h->peer_thr.push_back(reinterpret_cast<unsigned long long*>(pp));
    }
    h->peer_ipc = true;
    return PYROPE_OK;
}

int pyrope_index_threshold_exchange_close(pyrope_index* h) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::lock_guard<std::mutex> g(h->mu);
    CK(cudaStreamSynchronize(h->stream));
    if (h->last_stream) CK(cudaStreamSynchronize(h->last_stream));
    for (unsigned long long* pp : h->peer_thr) if (h->peer_ipc) cudaIpcCloseMemHandle(pp);
    h->peer_thr.clear();  // this rank's own array stays allocated: peers may still write into it
    return PYROPE_OK;
}

int pyrope_index_threshold_exchange_epoch(pyrope_index* h, uint32_t epoch) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (epoch == 0) return fail(PYROPE_ERR_INVALID_ARG, "epoch 0 is reserved (an empty word)");
    std::lock_guard<std::mutex> g(h->mu);
    h->thr_epoch = epoch;
    h->thr_epoch_set = true;
    return PYROPE_OK;
}

int pyrope_index_is_built(pyrope_index* h, int* out) {
    if (!h || !out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    *out = h->built ? 1 : 0;
    return PYROPE_OK;
}

int pyrope_index_get_centroids(pyrope_index* h, float* centroids_out, int* n_out) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::lock_guard<std::mutex> g(h->mu);
    int n = h->built ? h->nc : 0;
    if (n_out) *n_out = n;
    if (centroids_out && n > 0)
        CK(cudaMemcpy(centroids_out, h->centroids.p, sizeof(float) * (size_t)n * h->dim, cudaMemcpyDeviceToHost));
    return PYROPE_OK;
}

int pyrope_index_get_codebooks(pyrope_index* h, float* codebooks_out, int32_t* ksub_out) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (h->kind != PYROPE_IVF_PQ) return fail(PYROPE_ERR_INVALID_STATE, "not an IVF_PQ index");
    std::lock_guard<std::mutex> g(h->mu);
    if (h->ksub.empty()) return fail(PYROPE_ERR_INVALID_STATE, "PQ not trained");
    if (codebooks_out)
        CK(cudaMemcpy(codebooks_out, h->codebook.p, sizeof(float) * (size_t)h->m * h->k * h->sub, cudaMemcpyDeviceToHost));
    if (ksub_out) memcpy(ksub_out, h->ksub.data(), sizeof(int32_t) * (size_t)h->m);
    return PYROPE_OK;
}

int pyrope_index_get_lists(pyrope_index* h, int64_t* offsets_out, int64_t* rows_out, uint8_t* codes_out, int64_t* total_out) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::lock_guard<std::mutex> g(h->mu);
    if (!h->built) {
        if (total_out) *total_out = 0;
        return PYROPE_OK;
    }
    if (total_out) *total_out = h->lists.total;
    if (offsets_out) memcpy(offsets_out, h->lists.off_h.data(), sizeof(int64_t) * ((size_t)h->nc + 1));
    if (rows_out && h->lists.total)
        CK(cudaMemcpy(rows_out, h->lists.rows.p, sizeof(int64_t) * (size_t)h->lists.total, cudaMemcpyDeviceToHost));
    if (codes_out && h->lists.total && h->kind == PYROPE_IVF_PQ)
        CK(cudaMemcpy(codes_out, h->lists.payload.p, (size_t)h->lists.total * h->m, cudaMemcpyDeviceToHost));
    return PYROPE_OK;
}

// ---- snapshot / load (IVectorIndex.Snapshot / Load; DeltaVectorIndex.cs:160-212 writes tmp-then-move) -------
// Binary, little-endian, self-describing enough to refuse a mismatched index.  The reference's formats are JSON
// (BruteForce / IVF_FLAT) or a no-op (IVF_PQ, IvfPqVectorIndex.cs:228-229); a drop-in only has to round-trip
// its own state, which this does for all three kinds, trained codebooks and inverted lists included.
}  // extern "C"
namespace {
struct SnapIO {
    FILE* f = nullptr;
    bool ok = true;
    bool bounded = false;      // reading: `remaining` = bytes left in the file, no length field may exceed it
    uint64_t remaining = 0;
    uint64_t last_bytes = 0;   // byte count of the most recent rdev()
    std::vector<unsigned char> stage;
    void w(const void* p, size_t n) { if (ok && n && fwrite(p, 1, n, f) != n) ok = false; }
    void r(void* p, size_t n) {
        if (bounded) { if (n > remaining) { ok = false; return; } remaining -= n; }
        if (ok && n && fread(p, 1, n, f) != n) ok = false;
    }
    template <typename T> void wv(T v) { w(&v, sizeof v); }
    template <typename T> T rv() { T v{}; r(&v, sizeof v); return v; }
    template <typename T> void wvec(const std::vector<T>& v) { wv<uint64_t>(v.size()); w(v.data(), sizeof(T) * v.size()); }
    template <typename T> void rvec(std::vector<T>& v) {
        uint64_t n = rv<uint64_t>();
        if (!ok || n > ((uint64_t)1 << 40) || (bounded && n * sizeof(T) > remaining)) { ok = false; return; }
        v.resize((size_t)n);
        r(v.data(), sizeof(T) * v.size());
    }
    // device array <-> file through a 64 MiB host stage
    int wdev(const void* d, size_t bytes) {
        wv<uint64_t>(bytes);
        stage.resize(std::min<size_t>(bytes, (size_t)64 << 20));
        for (size_t o = 0; o < bytes; o += stage.size()) {
            size_t n = std::min(stage.size(), bytes - o);
            CK(cudaMemcpy(stage.data(), (const char*)d + o, n, cudaMemcpyDeviceToHost));
            w(stage.data(), n);
        }
        return PYROPE_OK;
    }
    int rdev(DevBuf& b, cudaStream_t st) {
        uint64_t bytes = rv<uint64_t>();
        last_bytes = 0;
        if (!ok || bytes > ((uint64_t)1 << 42) || (bounded && bytes > remaining)) { ok = false; return PYROPE_OK; }
        last_bytes = bytes;
        if (bytes == 0) return PYROPE_OK;
        TRY(b.ensure((size_t)bytes, 0, st, true));
        stage.resize(std::min<size_t>((size_t)bytes, (size_t)64 << 20));
        for (size_t o = 0; o < bytes; o += stage.size()) {
            size_t n = std::min(stage.size(), (size_t)bytes - o);
            r(stage.data(), n);
            if (!ok) return PYROPE_OK;
            CK(cudaMemcpy((char*)b.p + o, stage.data(), n, cudaMemcpyHostToDevice));
        }
        return PYROPE_OK;
    }
};
constexpr char kSnapMagic[8] = {'P', 'Y', 'R', 'G', 'P', 'U', '0', '1'};
}  // namespace
extern "C" {

int pyrope_index_snapshot(pyrope_index* h, const char* path) {
    if (!h || !path || !*path) return fail(PYROPE_ERR_INVALID_ARG, "Path cannot be empty");
    std::lock_guard<std::mutex> g(h->mu);
    CK(cudaStreamSynchronize(h->stream));
    if (h->last_stream) CK(cudaStreamSynchronize(h->last_stream));
    const std::string tmp = std::string(path) + ".tmp";
    SnapIO io;
    io.f = fopen(tmp.c_str(), "wb");
    if (!io.f) return fail(PYROPE_ERR_INVALID_ARG, "cannot open %s for writing", tmp.c_str());
    int rc = PYROPE_OK;
    auto body = [&]() -> int {
        io.w(kSnapMagic, 8);
        io.wv<int32_t>(h->kind); io.wv<int32_t>(h->dim); io.wv<int32_t>(h->metric); io.wv<int32_t>(h->nlist);
        io.wv<int32_t>(h->m); io.wv<int32_t>(h->k); io.wv<int64_t>(h->next_row);
        const Segment& s = h->seg;
        io.wv<int64_t>(s.nslots); io.wv<int64_t>(s.live); io.wv<int64_t>(s.ndead);
        TRY(io.wdev(s.X.p, sizeof(float) * (size_t)s.nslots * h->dim));
        TRY(io.wdev(s.labels.p, sizeof(int64_t) * (size_t)s.nslots));
        io.wvec(s.dead_h); io.wvec(s.slot_row); io.wvec(s.free_stack);
        io.wv<int32_t>(h->built ? 1 : 0); io.wv<int32_t>(h->frozen ? 1 : 0); io.wv<int32_t>(h->nc);
        io.wv<int32_t>(h->shard_rank); io.wv<int32_t>(h->shard_world);
        const bool have_cent = h->nc > 0 && h->centroids.p;
        TRY(io.wdev(h->centroids.p, have_cent ? sizeof(float) * (size_t)h->nc * h->dim : 0));
        const bool have_cb = h->kind == PYROPE_IVF_PQ && h->codebook.p && !h->ksub.empty();
        TRY(io.wdev(h->codebook.p, have_cb ? sizeof(float) * (size_t)h->m * h->k * h->sub : 0));
        io.wvec(h->ksub);
        io.wv<int64_t>(h->built ? h->lists.total : 0);
        if (h->built) {
            io.wvec(h->lists.off_h);
            TRY(io.wdev(h->lists.rows.p, sizeof(int64_t) * (size_t)h->lists.total));
            TRY(io.wdev(h->lists.labels.p, sizeof(int64_t) * (size_t)h->lists.total));
            const size_t per = h->kind == PYROPE_IVF_FLAT ? sizeof(float) * (size_t)h->dim : (size_t)h->m;
            TRY(io.wdev(h->lists.payload.p, (size_t)h->lists.total * per));
            io.wvec(h->lists.dead_h);
        }
        return PYROPE_OK;
    };
    rc = body();
    const bool ok = io.ok && fclose(io.f) == 0;
    if (rc != PYROPE_OK) { remove(tmp.c_str()); return rc; }
    if (!ok) { remove(tmp.c_str()); return fail(PYROPE_ERR_INVALID_STATE, "short write to %s", tmp.c_str()); }
    if (rename(tmp.c_str(), path) != 0) { remove(tmp.c_str()); return fail(PYROPE_ERR_INVALID_STATE, "cannot move %s into place", tmp.c_str()); }
    return PYROPE_OK;
}

// Everything a snapshot holds, parsed into temporaries: pyrope_index_load validates the WHOLE file against the
// index's shape (byte counts against nslots / dim / list_total / nc, offsets monotone and ending at list_total, row
// ordinals inside [0, next_row), counters consistent with the flags) and only then swaps it into the live index, so
// a truncated or corrupt file leaves the index exactly as it was.
}  // extern "C"
namespace {
struct LoadedSnapshot {
    int32_t nlist = 0;
    int64_t next_row = 0, nslots = 0, live = 0, ndead = 0;
    DevBuf X, labels, centroids, codebook, list_rows, list_labels, list_payload;
    std::vector<uint8_t> dead_h, list_dead_h;
    std::vector<int64_t> slot_row, free_stack, list_off_h;
    std::vector<int32_t> ksub;
    bool built = false, frozen = false;
    int32_t nc = 0, shard_rank = 0, shard_world = 1;
    int64_t list_total = 0;
};

// host copy of a device int64 array, checked to lie in [lo, hi) (allow_neg1: -1 is also fine)
int check_i64_range(const DevBuf& b, int64_t n, int64_t lo, int64_t hi, bool allow_neg1, const char* what) {
    std::vector<int64_t> v((size_t)std::min<int64_t>(n, (int64_t)1 << 22));
    for (int64_t o = 0; o < n; o += (int64_t)v.size()) {
        const int64_t c = std::min<int64_t>((int64_t)v.size(), n - o);
        CK(cudaMemcpy(v.data(), b.as<int64_t>() + o, sizeof(int64_t) * (size_t)c, cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < c; ++i) {
            const int64_t x = v[(size_t)i];
            if (!((x >= lo && x < hi) || (allow_neg1 && x == -1)))
                return fail(PYROPE_ERR_INVALID_ARG, "corrupt snapshot: %s[%lld] = %lld out of range", what, (long long)(o + i), (long long)x);
        }
    }
    return PYROPE_OK;
}

int parse_snapshot(const Index* h, SnapIO& io, const char* path, LoadedSnapshot& L, cudaStream_t st) {
    auto bad = [&](const char* what) { return fail(PYROPE_ERR_INVALID_ARG, "corrupt or truncated snapshot %s: %s", path, what); };
    char magic[8];
    io.r(magic, 8);
    if (!io.ok || memcmp(magic, kSnapMagic, 8) != 0) return fail(PYROPE_ERR_INVALID_ARG, "%s is not a pyrope_gpu snapshot", path);
    const int kind = io.rv<int32_t>(), dim = io.rv<int32_t>(), metric = io.rv<int32_t>();
    L.nlist = io.rv<int32_t>();
    const int m = io.rv<int32_t>(), k = io.rv<int32_t>();
    if (!io.ok) return bad("header");
    if (kind != h->kind || metric != h->metric || m != h->m || k != h->k) return fail(PYROPE_ERR_INVALID_ARG, "snapshot is of a different index type");
    if (dim != h->dim) return fail(PYROPE_ERR_DIMENSION, "Vector dimension mismatch");
    L.next_row = io.rv<int64_t>();
    L.nslots = io.rv<int64_t>(); L.live = io.rv<int64_t>(); L.ndead = io.rv<int64_t>();
    if (!io.ok || L.next_row < 0 || L.nslots < 0 || L.live < 0 || L.ndead < 0 || L.live + L.ndead != L.nslots ||
        L.nslots > ((int64_t)1 << 40) / std::max(dim, 1))
        return bad("row counters");
    const bool ivf = kind != PYROPE_FLAT;
    if (ivf ? L.nslots > L.next_row : L.nslots != L.next_row) return bad("more slots than rows ever added");
    TRY(io.rdev(L.X, st));
    if (!io.ok || io.last_bytes != sizeof(float) * (uint64_t)L.nslots * dim) return bad("row vectors");
    TRY(io.rdev(L.labels, st));
    if (!io.ok || io.last_bytes != sizeof(int64_t) * (uint64_t)L.nslots) return bad("row labels");
    io.rvec(L.dead_h); io.rvec(L.slot_row); io.rvec(L.free_stack);
    if (!io.ok || (int64_t)L.dead_h.size() != L.nslots) return bad("tombstone flags");
    int64_t nd = 0;
    for (uint8_t b : L.dead_h) nd += b ? 1 : 0;
    if (nd != L.ndead) return bad("tombstone count");
    if (ivf) {
        if ((int64_t)L.slot_row.size() != L.nslots || (int64_t)L.free_stack.size() != L.ndead) return bad("buffer slot tables");
        for (int64_t i = 0; i < L.nslots; ++i) {
            const int64_t r = L.slot_row[(size_t)i];
            if (L.dead_h[(size_t)i] ? r != -1 : (r < 0 || r >= L.next_row)) return bad("slot -> row table");
        }
        std::vector<uint8_t> seen((size_t)L.nslots, 0);
        for (int64_t sl : L.free_stack) {
            if (sl < 0 || sl >= L.nslots || !L.dead_h[(size_t)sl] || seen[(size_t)sl]) return bad("free-slot stack");
            seen[(size_t)sl] = 1;
        }
    } else if (!L.slot_row.empty() || !L.free_stack.empty()) {
        return bad("slot tables on a FLAT index");
    }
    L.built = io.rv<int32_t>() != 0; L.frozen = io.rv<int32_t>() != 0; L.nc = io.rv<int32_t>();
    L.shard_rank = io.rv<int32_t>(); L.shard_world = io.rv<int32_t>();
    if (!io.ok || L.nc < 0 || L.shard_world < 1 || L.shard_rank < 0 || L.shard_rank >= L.shard_world) return bad("build header");
    if (!ivf && (L.built || L.nc != 0)) return bad("inverted lists on a FLAT index");
    if (L.built && L.nc <= 0) return bad("built without centroids");
    TRY(io.rdev(L.centroids, st));
    if (!io.ok || (io.last_bytes != 0 && io.last_bytes != sizeof(float) * (uint64_t)L.nc * dim) || (L.built && io.last_bytes == 0))
        return bad("centroids");
    if (io.last_bytes == 0 && L.nc != 0 && !L.built) L.nc = 0;
    TRY(io.rdev(L.codebook, st));
    const uint64_t cb_bytes = kind == PYROPE_IVF_PQ ? sizeof(float) * (uint64_t)h->m * h->k * h->sub : 0;
    if (!io.ok || (io.last_bytes != 0 && io.last_bytes != cb_bytes)) return bad("PQ codebooks");
    const bool have_cb = io.last_bytes != 0;
    io.rvec(L.ksub);
    if (!io.ok || !(L.ksub.empty() || (kind == PYROPE_IVF_PQ && (int)L.ksub.size() == h->m))) return bad("codewords per subspace");
    for (int32_t ks : L.ksub)
        if (ks < 1 || ks > h->k) return bad("codewords per subspace");
    if (kind == PYROPE_IVF_PQ && (L.built || !L.ksub.empty()) && (!have_cb || L.ksub.empty())) return bad("PQ codebooks missing");
    L.list_total = io.rv<int64_t>();
    if (!io.ok || L.list_total < 0 || L.list_total > L.next_row || (!L.built && L.list_total != 0)) return bad("list total");
    if (L.built) {
        io.rvec(L.list_off_h);
        if (!io.ok || (int64_t)L.list_off_h.size() != (int64_t)L.nc + 1 || L.list_off_h[0] != 0 ||
            L.list_off_h[(size_t)L.nc] != L.list_total)
            return bad("list offsets");
        for (int c = 0; c < L.nc; ++c)
            if (L.list_off_h[(size_t)c + 1] < L.list_off_h[(size_t)c]) return bad("list offsets not monotone");
        TRY(io.rdev(L.list_rows, st));
        if (!io.ok || io.last_bytes != sizeof(int64_t) * (uint64_t)L.list_total) return bad("list rows");
        TRY(io.rdev(L.list_labels, st));
        if (!io.ok || io.last_bytes != sizeof(int64_t) * (uint64_t)L.list_total) return bad("list labels");
        TRY(io.rdev(L.list_payload, st));
        const uint64_t per = kind == PYROPE_IVF_FLAT ? sizeof(float) * (uint64_t)dim : (uint64_t)h->m;
        if (!io.ok || io.last_bytes != per * (uint64_t)L.list_total) return bad("list vectors / codes");
        io.rvec(L.list_dead_h);
        if (!io.ok || !(L.list_dead_h.empty() || (int64_t)L.list_dead_h.size() == L.list_total)) return bad("list tombstones");
        for (uint8_t b : L.list_dead_h)
            if (b > 3) return bad("list tombstones");
        if (L.list_total) TRY(check_i64_range(L.list_rows, L.list_total, 0, L.next_row, false, "list_rows"));
        if (kind == PYROPE_IVF_PQ && L.list_total) {  // a code byte indexes its sub-codebook: ksub <= k <= 256 entries, zero padded to k
            // (every byte value < k is addressable; k = 256 needs no check)
        }
    }
    if (!io.ok) return bad("short read");
    return PYROPE_OK;
}

// Load: everything that can fail (parse, validation, every device allocation) stages the file aside, so a truncated or
// corrupt file or an OOM leaves the index as it was.  The sharded index prepares every shard before it installs any
// (pyrope_sharded_load: all or nothing over N devices).
int load_prepare(const Index& h, const char* path, Staged& S) {
    CK(cudaStreamSynchronize(h.stream));
    if (h.last_stream) CK(cudaStreamSynchronize(h.last_stream));
    SnapIO io;
    io.f = fopen(path, "rb");
    if (!io.f) return fail(PYROPE_ERR_NOT_FOUND, "Snapshot file not found: %s", path);  // FileNotFoundException
    if (fseek(io.f, 0, SEEK_END) == 0) { io.remaining = (uint64_t)std::max<long>(ftell(io.f), 0); io.bounded = true; }
    rewind(io.f);
    cudaStream_t st = h.stream;
    LoadedSnapshot L;
    int rc = parse_snapshot(&h, io, path, L, st);
    fclose(io.f);
    if (rc != PYROPE_OK) return rc;

    const int dim = h.dim;
    Segment& ns = S.seg;
    ns.dim = dim; ns.cosine = h.seg.cosine; ns.reuse_slots = h.seg.reuse_slots;
    TRY(ns.reserve(std::max<int64_t>(L.nslots, 1), st, true));
    if (L.nslots) {
        CK(cudaMemcpyAsync(ns.X.p, L.X.p, sizeof(float) * (size_t)L.nslots * dim, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(ns.labels.p, L.labels.p, sizeof(int64_t) * (size_t)L.nslots, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(ns.dead.p, L.dead_h.data(), (size_t)L.nslots, cudaMemcpyHostToDevice, st));
        if (ns.cosine) CK(launch_row_norms_exact(ns.X.as<float>(), L.nslots, dim, dim, ns.norms.as<float>(), st));
    }
    ns.nslots = L.nslots; ns.live = L.live; ns.ndead = L.ndead;
    ns.dead_h.swap(L.dead_h); ns.slot_row.swap(L.slot_row); ns.free_stack.swap(L.free_stack);
    IvfLists& T = S.lists;
    if (L.built) {
        T.total = L.list_total;
        T.rows = std::move(L.list_rows);
        T.labels = std::move(L.list_labels);
        T.payload = std::move(L.list_payload);
        T.off_h.swap(L.list_off_h);
        TRY(T.off.ensure(sizeof(int64_t) * T.off_h.size(), 0, st, true));
        CK(cudaMemcpyAsync(T.off.p, T.off_h.data(), sizeof(int64_t) * T.off_h.size(), cudaMemcpyHostToDevice, st));
        for (int c = 0; c < L.nc; ++c) T.max_len = std::max(T.max_len, T.off_h[(size_t)c + 1] - T.off_h[(size_t)c]);
        if (!L.list_dead_h.empty()) {
            T.dead_h.swap(L.list_dead_h);
            TRY(T.dead.ensure((size_t)std::max<int64_t>(T.total, 1), 0, st, true));
            CK(cudaMemcpyAsync(T.dead.p, T.dead_h.data(), T.dead_h.size(), cudaMemcpyHostToDevice, st));
            for (uint8_t b : T.dead_h) T.ndead += b ? 1 : 0;
        }
        TRY(S.cnorms.ensure(sizeof(float) * (size_t)std::max(L.nc, 1), 0, st, true));
        if (h.metric == kCosine) {
            CK(launch_row_norms_exact(L.centroids.as<float>(), L.nc, dim, dim, S.cnorms.as<float>(), st));
            if (h.kind == PYROPE_IVF_FLAT && T.total) {
                TRY(T.norms.ensure(sizeof(float) * (size_t)T.total, 0, st, true));
                CK(launch_row_norms_exact(T.payload.as<float>(), T.total, dim, dim, T.norms.as<float>(), st));
            }
        }
    }
    CK(cudaStreamSynchronize(st));
    S.quantiser = true;
    S.centroids = std::move(L.centroids);
    S.codebook = std::move(L.codebook);
    S.ksub.swap(L.ksub);
    S.nc = L.nc; S.built = L.built; S.frozen = L.frozen;
    S.load = true;
    S.nlist = L.nlist;
    S.next_row = L.next_row;
    S.shard_rank = L.shard_rank; S.shard_world = L.shard_world;
    S.noop = false;
    return PYROPE_OK;
}

// the first half of pyrope_internal_index_prepare_*: a Staged on the heap that the caller commits or discards
template <typename Prepare>
int prepare_detached(pyrope_index* h, void** staged_out, pyrope_internal_staged_info* info, Prepare prepare) {
    if (!h || !staged_out) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    *staged_out = nullptr;
    std::lock_guard<std::mutex> g(h->mu);
    std::unique_ptr<Staged> S(new (std::nothrow) Staged(*h));
    if (!S) return fail(PYROPE_ERR_OOM, "out of host memory");
    TRY(prepare(*h, *S));
    if (info) {
        info->n_moved = (int64_t)S->moved.size();
        info->moved = S->moved.data();
        info->shard_rank = S->shard_rank;
        info->shard_world = S->shard_world;
        info->next_row = S->next_row;
    }
    *staged_out = S.release();
    return PYROPE_OK;
}
}  // namespace
extern "C" {

int pyrope_index_load(pyrope_index* h, const char* path) {
    if (!h || !path || !*path) return fail(PYROPE_ERR_INVALID_ARG, "Path cannot be empty");
    std::lock_guard<std::mutex> g(h->mu);
    Staged S(*h);
    TRY(load_prepare(*h, path, S));
    install(h, S);
    return PYROPE_OK;
}

int pyrope_internal_index_prepare_build(pyrope_index* h, void** staged_out, pyrope_internal_staged_info* info) {
    return prepare_detached(h, staged_out, info, build_prepare);
}

int pyrope_internal_index_prepare_extend(pyrope_index* h, void** staged_out, pyrope_internal_staged_info* info) {
    return prepare_detached(h, staged_out, info, extend_prepare);
}

int pyrope_internal_index_prepare_load(pyrope_index* h, const char* path, void** staged_out, pyrope_internal_staged_info* info) {
    if (!path || !*path) return fail(PYROPE_ERR_INVALID_ARG, "Path cannot be empty");
    return prepare_detached(h, staged_out, info, [path](const Index& x, Staged& S) { return load_prepare(x, path, S); });
}

void pyrope_internal_index_commit(pyrope_index* h, void* staged) {
    std::unique_ptr<Staged> S(static_cast<Staged*>(staged));
    std::lock_guard<std::mutex> g(h->mu);
    install(h, *S);
}

void pyrope_internal_index_discard(void* staged) { delete static_cast<Staged*>(staged); }

// header peek for the string-id layer: rows ever added according to the snapshot (validates the magic only)
int pyrope_internal_snapshot_next_row(const char* path, int64_t* next_row_out) {
    FILE* f = fopen(path, "rb");
    if (!f) return fail(PYROPE_ERR_NOT_FOUND, "Snapshot file not found: %s", path);
    char magic[8];
    int32_t hdr[6];
    int64_t nr = -1;
    const bool ok = fread(magic, 1, 8, f) == 8 && memcmp(magic, kSnapMagic, 8) == 0 &&
                    fread(hdr, 4, 6, f) == 6 && fread(&nr, 8, 1, f) == 1 && nr >= 0;
    fclose(f);
    if (!ok) return fail(PYROPE_ERR_INVALID_ARG, "%s is not a pyrope_gpu snapshot", path);
    *next_row_out = nr;
    return PYROPE_OK;
}

int pyrope_index_stats(pyrope_index* h, int64_t* live_rows, int64_t* buffer_rows, int* dim, int* metric) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (live_rows) *live_rows = h->seg.live + (h->built ? h->lists.total - h->lists.ndead : 0);
    if (buffer_rows) *buffer_rows = h->seg.live;
    if (dim) *dim = h->dim;
    if (metric) *metric = h->metric;
    return PYROPE_OK;
}

int pyrope_index_search_batch_device(pyrope_index* h, int64_t nq, const float* dQ, int topk, int64_t max_scans,
                                     int nprobe, float* d_scores, int64_t* d_rows, int32_t* d_counts, void* stream) {
    TRY(validate_search(h, nq, dQ, topk));
    if (nq == 0) return PYROPE_OK;
    std::lock_guard<std::mutex> g(h->mu);
    if (h->kind == PYROPE_IVF_FLAT && max_scans >= 0 && h->lists.ndead > 0) TRY(compact_lists(h));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    TRY(search_device(h, nq, dQ, topk, max_scans, nprobe, d_scores, d_rows, d_counts, st));
    if (!stream) CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

int pyrope_index_coarse_probe_device(pyrope_index* h, int64_t nq, const float* dQ, int nprobe, int64_t* d_probes_out,
                                     void* stream) {
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (nq < 0 || (nq > 0 && (!dQ || !d_probes_out))) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    if (h->kind == PYROPE_FLAT) return fail(PYROPE_ERR_INVALID_STATE, "FLAT has no coarse stage");
    if (nq == 0) return PYROPE_OK;
    std::lock_guard<std::mutex> g(h->mu);
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    TRY(search_device(h, nq, dQ, 1, -1, nprobe, nullptr, nullptr, nullptr, st, nullptr, d_probes_out));
    if (!stream) CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

int pyrope_index_search_batch_probed_device(pyrope_index* h, int64_t nq, const float* dQ, int topk, int64_t max_scans,
                                            int nprobe, const int64_t* d_probes, float* d_scores, int64_t* d_rows,
                                            int32_t* d_counts, void* stream) {
    TRY(validate_search(h, nq, dQ, topk));
    if (h->kind == PYROPE_FLAT) return fail(PYROPE_ERR_INVALID_STATE, "FLAT has no coarse stage");
    if (!d_probes) return fail(PYROPE_ERR_INVALID_ARG, "probes is null");
    if (nq == 0) return PYROPE_OK;
    std::lock_guard<std::mutex> g(h->mu);
    if (h->kind == PYROPE_IVF_FLAT && max_scans >= 0 && h->lists.ndead > 0) TRY(compact_lists(h));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    TRY(search_device(h, nq, dQ, topk, max_scans, nprobe, d_scores, d_rows, d_counts, st, d_probes, nullptr));
    if (!stream) CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

int pyrope_index_search_batch(pyrope_index* h, int64_t nq, const float* Q, int topk, int64_t max_scans, int nprobe,
                              float* scores_out, int64_t* rows_out, int32_t* counts_out) {
    TRY(validate_search(h, nq, Q, topk));
    if (nq == 0) return PYROPE_OK;
    if (!scores_out || !rows_out || !counts_out) return fail(PYROPE_ERR_INVALID_ARG, "output buffer is null");
    std::lock_guard<std::mutex> g(h->mu);
    if (h->kind == PYROPE_IVF_FLAT && max_scans >= 0 && h->lists.ndead > 0) TRY(compact_lists(h));
    cudaStream_t st = h->stream;
    Workspace& ws = h->ws;
    const int kk = std::max(topk, 1);
    TRY(ws.hq.ensure(sizeof(float) * (size_t)nq * h->dim, 0, st));
    TRY(ws.hs.ensure(sizeof(float) * (size_t)nq * kk, 0, st));
    TRY(ws.hl.ensure(sizeof(int64_t) * (size_t)nq * kk, 0, st));
    TRY(ws.hc.ensure(sizeof(int32_t) * (size_t)nq, 0, st));
    CK(cudaMemcpyAsync(ws.hq.p, Q, sizeof(float) * (size_t)nq * h->dim, cudaMemcpyHostToDevice, st));
    TRY(search_device(h, nq, ws.hq.as<float>(), topk, max_scans, nprobe, ws.hs.as<float>(), ws.hl.as<int64_t>(),
                      ws.hc.as<int32_t>(), st));
    if (topk > 0) {
        CK(cudaMemcpyAsync(scores_out, ws.hs.p, sizeof(float) * (size_t)nq * topk, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(rows_out, ws.hl.p, sizeof(int64_t) * (size_t)nq * topk, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaMemcpyAsync(counts_out, ws.hc.p, sizeof(int32_t) * (size_t)nq, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

int pyrope_index_last_search_ms(pyrope_index* h, float* out4) {
    if (!h || !out4) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    std::lock_guard<std::mutex> g(h->mu);
    out4[0] = out4[1] = out4[2] = out4[3] = 0.f;
    if (!h->ev_valid) return PYROPE_OK;
    CK(cudaEventSynchronize(h->ev[3]));
    CK(cudaEventElapsedTime(&out4[0], h->ev[0], h->ev[3]));
    CK(cudaEventElapsedTime(&out4[1], h->ev[0], h->ev[1]));
    CK(cudaEventElapsedTime(&out4[2], h->ev[1], h->ev[2]));
    CK(cudaEventElapsedTime(&out4[3], h->ev[2], h->ev[3]));
    return PYROPE_OK;
}

int pyrope_index_last_search_kernel(pyrope_index* h, float* ms_out, const char** name_out) {
    if (!h || !ms_out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    std::lock_guard<std::mutex> g(h->mu);
    *ms_out = 0.f;
    if (name_out) *name_out = h->dom_kernel;
    if (!h->evk_valid) return PYROPE_OK;
    CK(cudaEventSynchronize(h->evk[1]));
    CK(cudaEventElapsedTime(ms_out, h->evk[0], h->evk[1]));
    return PYROPE_OK;
}

int pyrope_index_last_search_launches(pyrope_index* h, int* out) {
    if (!h || !out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    *out = h->last_launches;
    return PYROPE_OK;
}

int pyrope_index_last_search_scanned(pyrope_index* h, int64_t* codes_out) {
    if (!h || !codes_out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    std::lock_guard<std::mutex> g(h->mu);
    *codes_out = 0;
    if (h->lm_nq <= 0 || !h->ws.lm.p) return PYROPE_OK;
    unsigned long long v = 0;
    if (h->kind == PYROPE_IVF_FLAT)
        CK(ivfflat_lm_scanned_rows(h->ws.lm.p, h->lm_nq, h->lm_P, h->lm_k, h->nc, &v, h->last_stream ? h->last_stream : h->stream));
    else
        CK(ivfpq_lm_scanned_codes(h->ws.lm.p, h->lm_nq, h->lm_P, h->lm_k, h->nc, h->dim, h->lists.max_len, &v,
                                  h->last_stream ? h->last_stream : h->stream));
    *codes_out = (int64_t)v;
    return PYROPE_OK;
}

int pyrope_topk_merge_dedupe_device(int64_t nq, int parts, int k_in, int k_out, const float* d_scores, const int64_t* d_rows,
                                    float* d_scores_out, int64_t* d_rows_out, int32_t* d_counts_out, int dedupe, void* stream) {
    if (nq < 0 || parts <= 0 || k_in <= 0 || k_out <= 0) return fail(PYROPE_ERR_INVALID_ARG, "bad merge shape");
    if ((int64_t)parts * k_in > kMergeMaxCandidates)
        return fail(PYROPE_ERR_UNSUPPORTED, "parts*k_in = %lld exceeds %d", (long long)parts * k_in, kMergeMaxCandidates);
    CK(launch_merge_pairs(nq, parts, k_in, k_out, d_scores, d_rows, nq * (int64_t)k_in, k_in, d_scores_out, d_rows_out,
                          d_counts_out, (cudaStream_t)stream, dedupe != 0));
    if (!stream) CK(cudaStreamSynchronize(nullptr));
    return PYROPE_OK;
}

int pyrope_topk_merge_device(int64_t nq, int parts, int k_in, int k_out, const float* d_scores, const int64_t* d_rows,
                             float* d_scores_out, int64_t* d_rows_out, int32_t* d_counts_out, void* stream) {
    return pyrope_topk_merge_dedupe_device(nq, parts, k_in, k_out, d_scores, d_rows, d_scores_out, d_rows_out, d_counts_out, 0, stream);
}

// ---- Head+Tail on device (DeltaVectorIndex.cs) ------------------------------------------------------
}  // extern "C"

struct pyrope_delta {
    pyrope_index* head = nullptr;
    pyrope_index* tail = nullptr;    // single-device tail, or
    pyrope_sharded* stail = nullptr;  // a tail sharded over the devices of the box (pyrope_delta_create_sharded)
    int tail_devices = 1;
    std::mutex mu;
    DevBuf ps, pl, pc, q, os, ol, oc;  // partial (head | tail) results, staged queries, merged outputs
    DevBuf kq;                         // per-query topK of pyrope_delta_search_batch_topk
    cudaEvent_t q_ready = nullptr;     // sharded tail: the queries are in place on the head's stream
};

namespace {

// DeltaVectorIndex.Search:76-122 for nq queries: head top-k, tail top-k (same options, :85,88), merge by id with
// the head's copy winning, descending, Take(topK) — one stream, no host round trip between the three stages.
// d_kq (nullable, device [nq], every entry <= topk): query i asked for d_kq[i].  Both sides still run once at topk, and
// the merge keeps only each side's first d_kq[i] entries.  Cutting the merged list at d_kq[i] instead would be wrong:
// an id the head shares with the tail's top d_kq[i] would let the tail's (d_kq[i]+1)-th entry into the result.
int delta_search_device(pyrope_delta* d, int64_t nq, const float* dQ, int topk, int64_t max_scans, int nprobe,
                        float* d_scores, int64_t* d_labels, int32_t* d_counts, cudaStream_t st,
                        const int32_t* d_kq = nullptr) {
    Index* hd = d->head;
    Index* tl = d->tail;
    const size_t per = (size_t)nq * topk;
    TRY(d->ps.ensure(sizeof(float) * 2 * per, 0, st));
    TRY(d->pl.ensure(sizeof(int64_t) * 2 * per, 0, st));
    TRY(d->pc.ensure(sizeof(int32_t) * 2 * (size_t)nq, 0, st));
    if (d->stail) CK(cudaEventRecord(d->q_ready, st));  // before the head's search: the tail does not wait for it
    {
        std::lock_guard<std::mutex> g(hd->mu);
        TRY(search_device(hd, nq, dQ, topk, max_scans, nprobe, d->ps.as<float>(), d->pl.as<int64_t>(),
                          d->pc.as<int32_t>(), st));
    }
    if (d->stail) {
        // The head's top-k is enqueued and overlaps the tail's coarse stage.  The sharded search merges the shards'
        // lists down to the tail's top k first: the reference asks the tail for topK (:88), so an id the head also
        // holds costs the result one tail entry, and a single merge of head and per-shard lists would refill that slot
        // with the tail's (k+1)-th.  An IVF_PQ tail ignores MaxScans (IvfPqVectorIndex.cs), an IVF_FLAT tail over
        // several devices refuses it (UNSUPPORTED, as pyrope_sharded_search_batch does).
        Index* t0 = nullptr;
        TRY(pyrope_sharded_shard(d->stail, 0, &t0, nullptr));
        TRY(pyrope_internal_sharded_search_device(d->stail, nq, dQ, topk, t0->kind == PYROPE_IVF_PQ ? -1 : max_scans,
                                                  nprobe, d->ps.as<float>() + per, d->pl.as<int64_t>() + per,
                                                  d->pc.as<int32_t>() + nq, d->q_ready));
    } else {
        std::lock_guard<std::mutex> g(tl->mu);
        if (tl->kind == PYROPE_IVF_FLAT && max_scans >= 0 && tl->lists.ndead > 0) TRY(compact_lists(tl));
        TRY(search_device(tl, nq, dQ, topk, max_scans, nprobe, d->ps.as<float>() + per, d->pl.as<int64_t>() + per,
                          d->pc.as<int32_t>() + nq, st));
    }
    CK(launch_merge_pairs(nq, 2, topk, topk, d->ps.as<float>(), d->pl.as<int64_t>(), (int64_t)per, topk, d_scores,
                          d_labels, d_counts, st, /*dedupe=*/true, d_kq));
    return PYROPE_OK;
}

// the head's and the tail's lists share one merge of at most kMergeMaxCandidates candidates
int delta_max_topk(const pyrope_delta* d) { return std::min(kMaxTopK, kMergeMaxCandidates / std::max(2, d->tail_devices)); }

int delta_validate(pyrope_delta* d, int64_t nq, const float* Q, int topk) {
    if (!d) return fail(PYROPE_ERR_INVALID_ARG, "delta handle is null");
    if (nq < 0 || (nq > 0 && !Q)) return fail(PYROPE_ERR_INVALID_ARG, "query is null");
    if (topk <= 0) return fail(PYROPE_ERR_OUT_OF_RANGE, "topK must be positive.");  // the FLAT head throws first
    const int lim = delta_max_topk(d);
    if (topk > lim) return fail(PYROPE_ERR_UNSUPPORTED, "topK %d exceeds the supported maximum %d", topk, lim);
    return PYROPE_OK;
}

// the tail's last search ran on the head's stream: do not leave it a handle the head may destroy first
void delta_forget_stream(pyrope_delta* d, cudaStream_t st) {
    if (d->tail && d->tail->last_stream == st) d->tail->last_stream = nullptr;
}

}  // namespace

extern "C" {

int pyrope_delta_create(pyrope_index* head, pyrope_index* tail, pyrope_delta** out) {
    if (!out) return fail(PYROPE_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    if (!head || !tail) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (head == tail) return fail(PYROPE_ERR_INVALID_ARG, "Head and Tail must be different indexes");
    if (head->dim != tail->dim) return fail(PYROPE_ERR_INVALID_ARG, "Head and Tail dimensions must match");
    if (head->metric != tail->metric) return fail(PYROPE_ERR_INVALID_ARG, "Head and Tail metrics must match");
    if (head->kind != PYROPE_FLAT) return fail(PYROPE_ERR_UNSUPPORTED, "the head must be a FLAT index");
    pyrope_delta* d = new (std::nothrow) pyrope_delta();
    if (!d) return fail(PYROPE_ERR_OOM, "out of host memory");
    d->head = head;
    d->tail = tail;
    *out = d;
    return PYROPE_OK;
}

int pyrope_delta_create_sharded(pyrope_index* head, pyrope_sharded* tail, pyrope_delta** out) {
    if (!out) return fail(PYROPE_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    if (!head || !tail) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    Index* t0 = nullptr;
    int dev0 = -1, n = 0;
    TRY(pyrope_sharded_shard(tail, 0, &t0, &dev0));
    TRY(pyrope_sharded_device_count(tail, &n));
    if (head == t0) return fail(PYROPE_ERR_INVALID_ARG, "Head and Tail must be different indexes");
    if (head->dim != t0->dim) return fail(PYROPE_ERR_INVALID_ARG, "Head and Tail dimensions must match");
    if (head->metric != t0->metric) return fail(PYROPE_ERR_INVALID_ARG, "Head and Tail metrics must match");
    if (head->kind != PYROPE_FLAT) return fail(PYROPE_ERR_UNSUPPORTED, "the head must be a FLAT index");
    if (head->device != dev0)
        return fail(PYROPE_ERR_INVALID_ARG, "the head lives on device %d, the sharded tail's first device is %d", head->device, dev0);
    if (t0->kind == PYROPE_FLAT) return fail(PYROPE_ERR_UNSUPPORTED, "a sharded tail must be IVF_FLAT or IVF_PQ");
    pyrope_delta* d = new (std::nothrow) pyrope_delta();
    if (!d) return fail(PYROPE_ERR_OOM, "out of host memory");
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(head->device);  // the event is recorded on the head's stream
    cudaError_t e = cudaEventCreateWithFlags(&d->q_ready, cudaEventDisableTiming);
    cudaSetDevice(cur);
    if (e != cudaSuccess) { delete d; return fail(PYROPE_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(e)); }
    d->head = head;
    d->stail = tail;
    d->tail_devices = n;
    *out = d;
    return PYROPE_OK;
}

int pyrope_delta_destroy(pyrope_delta* d) {
    if (!d) return PYROPE_OK;
    cudaStreamSynchronize(d->head->stream);
    delta_forget_stream(d, d->head->stream);
    if (d->q_ready) cudaEventDestroy(d->q_ready);
    delete d;
    return PYROPE_OK;
}

int pyrope_delta_search_batch_device(pyrope_delta* d, int64_t nq, const float* dQ, int topk, int64_t max_scans,
                                     int nprobe, float* d_scores, int64_t* d_labels, int32_t* d_counts, void* stream) {
    TRY(delta_validate(d, nq, dQ, topk));
    if (nq == 0) return PYROPE_OK;
    if (!d_scores || !d_labels) return fail(PYROPE_ERR_INVALID_ARG, "output buffer is null");
    std::lock_guard<std::mutex> g(d->mu);
    cudaStream_t st = stream ? (cudaStream_t)stream : d->head->stream;
    TRY(delta_search_device(d, nq, dQ, topk, max_scans, nprobe, d_scores, d_labels, d_counts, st));
    if (!stream) {
        CK(cudaStreamSynchronize(st));
        delta_forget_stream(d, st);
    }
    return PYROPE_OK;
}

}  // extern "C"

namespace {
// host queries in, host results out (stride topk); topks (nullable, host [nq], each <= topk): per-query topK
int delta_search_host(pyrope_delta* d, int64_t nq, const float* Q, int topk, const int32_t* topks, int64_t max_scans,
                      int nprobe, float* scores_out, int64_t* labels_out, int32_t* counts_out) {
    if (!scores_out || !labels_out || !counts_out) return fail(PYROPE_ERR_INVALID_ARG, "output buffer is null");
    std::lock_guard<std::mutex> g(d->mu);
    cudaStream_t st = d->head->stream;
    const int dim = d->head->dim;
    TRY(d->q.ensure(sizeof(float) * (size_t)nq * dim, 0, st));
    TRY(d->os.ensure(sizeof(float) * (size_t)nq * topk, 0, st));
    TRY(d->ol.ensure(sizeof(int64_t) * (size_t)nq * topk, 0, st));
    TRY(d->oc.ensure(sizeof(int32_t) * (size_t)nq, 0, st));
    CK(cudaMemcpyAsync(d->q.p, Q, sizeof(float) * (size_t)nq * dim, cudaMemcpyHostToDevice, st));
    if (topks) {
        TRY(d->kq.ensure(sizeof(int32_t) * (size_t)nq, 0, st));
        CK(cudaMemcpyAsync(d->kq.p, topks, sizeof(int32_t) * (size_t)nq, cudaMemcpyHostToDevice, st));
    }
    TRY(delta_search_device(d, nq, d->q.as<float>(), topk, max_scans, nprobe, d->os.as<float>(), d->ol.as<int64_t>(),
                            d->oc.as<int32_t>(), st, topks ? d->kq.as<int32_t>() : nullptr));
    CK(cudaMemcpyAsync(scores_out, d->os.p, sizeof(float) * (size_t)nq * topk, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(labels_out, d->ol.p, sizeof(int64_t) * (size_t)nq * topk, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(counts_out, d->oc.p, sizeof(int32_t) * (size_t)nq, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    delta_forget_stream(d, st);
    return PYROPE_OK;
}
}  // namespace

extern "C" {

int pyrope_delta_search_batch(pyrope_delta* d, int64_t nq, const float* Q, int topk, int64_t max_scans, int nprobe,
                              float* scores_out, int64_t* labels_out, int32_t* counts_out) {
    TRY(delta_validate(d, nq, Q, topk));
    if (nq == 0) return PYROPE_OK;
    return delta_search_host(d, nq, Q, topk, nullptr, max_scans, nprobe, scores_out, labels_out, counts_out);
}

int pyrope_delta_search_batch_topk(pyrope_delta* d, int64_t nq, const float* Q, const int32_t* topks, int64_t max_scans,
                                   int nprobe, float* scores_out, int64_t* labels_out, int32_t* counts_out) {
    if (nq > 0 && !topks) return fail(PYROPE_ERR_INVALID_ARG, "topks is null");
    int kmax = 1;
    for (int64_t i = 0; i < nq; ++i) {
        TRY(delta_validate(d, nq, Q, topks[i]));
        kmax = std::max(kmax, (int)topks[i]);
    }
    TRY(delta_validate(d, nq, Q, kmax));
    if (nq == 0) return PYROPE_OK;
    return delta_search_host(d, nq, Q, kmax, topks, max_scans, nprobe, scores_out, labels_out, counts_out);
}

// csrc/batcher.cu (internal): the dimension of a Head+Tail and the largest topK its search accepts
int pyrope_internal_delta_limits(pyrope_delta* d, int* dim_out, int* max_topk_out) {
    if (!d) return fail(PYROPE_ERR_INVALID_ARG, "delta handle is null");
    if (dim_out) *dim_out = d->head->dim;
    if (max_topk_out) *max_topk_out = delta_max_topk(d);
    return PYROPE_OK;
}

// csrc/batcher.cu (internal): FLAT / IVF_FLAT / IVF_PQ of an index (topK <= 0 is an error only on FLAT)
int pyrope_internal_index_kind(pyrope_index* h, int* kind_out) {
    if (!h || !kind_out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    *kind_out = h->kind;
    return PYROPE_OK;
}

}  // extern "C"

namespace {
// 1. of DeltaVectorIndex.Build: the head's live rows in scan order (bfHead.Scan(), DeltaVectorIndex.cs:133), gathered on
// the head's device into mx (n x dim) / ml (labels, also copied to the host as mlab).  Caller holds hd->mu.
int gather_head_rows(Index* hd, int64_t n, DevBuf& mx, DevBuf& ml, std::vector<int64_t>& mlab, cudaStream_t st) {
    const Segment& hs = hd->seg;
    const int dim = hd->dim;
    std::vector<int64_t> slots;
    slots.reserve((size_t)n);
    for (int64_t i = 0; i < hs.nslots; ++i)
        if (!hs.dead_h[(size_t)i]) slots.push_back(i);
    DevBuf idx;
    TRY(idx.ensure(sizeof(int64_t) * (size_t)n, 0, st, true));
    TRY(mx.ensure(sizeof(float) * (size_t)n * dim, 0, st, true));
    TRY(ml.ensure(sizeof(int64_t) * (size_t)n, 0, st, true));
    CK(cudaStreamSynchronize(hd->stream));
    CK(cudaMemcpyAsync(idx.p, slots.data(), sizeof(int64_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    CK(launch_gather_rows(hs.X.p, (int64_t)dim * 4, idx.as<int64_t>(), n, mx.p, st));
    CK(launch_gather_rows(hs.labels.p, 8, idx.as<int64_t>(), n, ml.p, st));
    mlab.resize((size_t)n);
    CK(cudaMemcpyAsync(mlab.data(), ml.p, sizeof(int64_t) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return PYROPE_OK;
}

// 2. of DeltaVectorIndex.Build: _tail.Add(id, vec) per row (:146) for n rows mx / ml (device, on the tail's device; labels
// also on the host as mlab): an id the tail already buffers is overwritten in place (Dictionary semantics,
// IvfFlatVectorIndex.cs:47 / IvfPqVectorIndex.cs:42); an id that sits in an inverted list is shadowed by the new buffer
// row until the tail's Build folds it in.  tail_rows_out (nullable): the tail row ordinal now holding each row.  Caller
// holds tl->mu with the tail's last search finished.
int tail_absorb(Index* tl, int64_t n, const float* mx, const int64_t* ml, const int64_t* mlab, int64_t* tail_rows_out) {
    cudaStream_t st = tl->stream;
    const int dim = tl->dim;
    std::vector<int64_t> order((size_t)n);  // moved rows sorted by label
    for (int64_t i = 0; i < n; ++i) order[(size_t)i] = i;
    std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return mlab[(size_t)a] < mlab[(size_t)b]; });
    std::vector<int64_t> sorted((size_t)n);
    for (int64_t i = 0; i < n; ++i) sorted[(size_t)i] = mlab[(size_t)order[(size_t)i]];
    std::vector<int64_t> target((size_t)n, -1);  // moved row -> tail buffer slot it overwrites
    DevBuf dsorted, where;
    Segment& ts = tl->seg;
    // both IVF searches skip a list entry whose id is buffered (seenIds, IvfFlatVectorIndex.cs:210, IvfPqVectorIndex.cs:170),
    // and an Extend that moves the buffered copy into the lists must find the entry it replaces flagged
    const bool lists_matter = tl->built && tl->kind != PYROPE_FLAT && tl->lists.total > 0;
    if (ts.live > 0 || lists_matter) {
        TRY(dsorted.ensure(sizeof(int64_t) * (size_t)n, 0, st, true));
        CK(cudaMemcpyAsync(dsorted.p, sorted.data(), sizeof(int64_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    }
    if (ts.live > 0) {
        TRY(where.ensure(sizeof(int64_t) * (size_t)ts.nslots, 0, st, true));
        CK(launch_find_labels(ts.labels.as<int64_t>(), ts.dead.as<uint8_t>(), ts.nslots, dsorted.as<int64_t>(), n,
                              where.as<int64_t>(), st));
        std::vector<int64_t> wh((size_t)ts.nslots);
        CK(cudaMemcpyAsync(wh.data(), where.p, sizeof(int64_t) * wh.size(), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (int64_t s = 0; s < ts.nslots; ++s)
            if (wh[(size_t)s] >= 0) target[(size_t)order[(size_t)wh[(size_t)s]]] = s;
    }
    if (lists_matter) {
        TRY(ensure_list_dead(tl));
        TRY(where.ensure(sizeof(int64_t) * (size_t)tl->lists.total, 0, st, true));
        CK(launch_find_labels(tl->lists.labels.as<int64_t>(), tl->lists.dead.as<uint8_t>(), tl->lists.total,
                              dsorted.as<int64_t>(), n, where.as<int64_t>(), st));
        std::vector<int64_t> wh((size_t)tl->lists.total);
        CK(cudaMemcpyAsync(wh.data(), where.p, sizeof(int64_t) * wh.size(), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        std::vector<int64_t> shadow;
        for (int64_t i = 0; i < tl->lists.total; ++i)
            if (wh[(size_t)i] >= 0) shadow.push_back(i);
        TRY(set_list_flag(tl, shadow, 2, true));
    }
    std::vector<int64_t> over_src, over_dst, app_src;
    for (int64_t i = 0; i < n; ++i) {
        if (target[(size_t)i] >= 0) { over_src.push_back(i); over_dst.push_back(target[(size_t)i]); }
        else app_src.push_back(i);
    }
    if (!over_src.empty()) {
        const int64_t no = (int64_t)over_src.size();
        DevBuf a, b, tmp;
        TRY(a.ensure(sizeof(int64_t) * (size_t)no, 0, st, true));
        TRY(b.ensure(sizeof(int64_t) * (size_t)no, 0, st, true));
        TRY(tmp.ensure(sizeof(float) * (size_t)no * dim, 0, st, true));
        CK(cudaMemcpyAsync(a.p, over_src.data(), sizeof(int64_t) * (size_t)no, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(b.p, over_dst.data(), sizeof(int64_t) * (size_t)no, cudaMemcpyHostToDevice, st));
        CK(launch_gather_rows(mx, (int64_t)dim * 4, a.as<int64_t>(), no, tmp.p, st));
        CK(launch_scatter_rows(tmp.p, (int64_t)dim * 4, b.as<int64_t>(), no, ts.X.p, st));
        if (ts.cosine)
            for (int64_t i = 0; i < no; ++i)
                CK(launch_row_norms_exact(ts.X.as<float>() + over_dst[(size_t)i] * dim, 1, dim, dim,
                                          ts.norms.as<float>() + over_dst[(size_t)i], st));
        ts.tc_dirty = true;
        CK(cudaStreamSynchronize(st));
        if (tl->kind == PYROPE_FLAT)
            for (int64_t i = 0; i < no; ++i) TRY(sq8_rows(tl, over_dst[(size_t)i], 1));
        if (tail_rows_out)
            for (int64_t i = 0; i < no; ++i)
                tail_rows_out[over_src[(size_t)i]] =
                    tl->kind == PYROPE_FLAT ? over_dst[(size_t)i] : ts.slot_row[(size_t)over_dst[(size_t)i]];
    }
    if (!app_src.empty()) {
        const int64_t na = (int64_t)app_src.size();
        const float* ax = mx;
        const int64_t* al = ml;
        DevBuf a, tx, tlab;
        if (na != n) {
            TRY(a.ensure(sizeof(int64_t) * (size_t)na, 0, st, true));
            TRY(tx.ensure(sizeof(float) * (size_t)na * dim, 0, st, true));
            TRY(tlab.ensure(sizeof(int64_t) * (size_t)na, 0, st, true));
            CK(cudaMemcpyAsync(a.p, app_src.data(), sizeof(int64_t) * (size_t)na, cudaMemcpyHostToDevice, st));
            CK(launch_gather_rows(mx, (int64_t)dim * 4, a.as<int64_t>(), na, tx.p, st));
            CK(launch_gather_rows(ml, 8, a.as<int64_t>(), na, tlab.p, st));
            CK(cudaStreamSynchronize(st));
            ax = tx.as<float>();
            al = tlab.as<int64_t>();
        }
        const int64_t first = tl->next_row;
        if (tl->kind != PYROPE_FLAT) tl->row_loc.resize((size_t)(first + na), -1);
        tl->next_row += na;
        const int64_t slot0 = ts.nslots;
        int r = seg_append(tl, na, ax, true, al, true, first);
        if (r != PYROPE_OK) { tl->next_row = first; return r; }
        if (tl->kind == PYROPE_FLAT) TRY(sq8_rows(tl, slot0, na));  // a FLAT tail with EnableQuantization
        if (tail_rows_out)
            for (int64_t i = 0; i < na; ++i) tail_rows_out[app_src[(size_t)i]] = first + i;
    }
    return PYROPE_OK;
}

// DeltaVectorIndex.Build :124-158 in two steps a caller can take apart: MOVE (head rows -> tail buffer, head tombstoned)
// and BUILD (the tail's Build, or with extend its Extend).  A host that keeps id tables updates them after the move
// whatever the build returns.
int delta_compact_impl(pyrope_delta* d, int64_t* moved_out, int64_t* tail_rows_out, bool do_move, bool do_build,
                       bool extend = false) {
    if (!d) return fail(PYROPE_ERR_INVALID_ARG, "delta handle is null");
    if (moved_out) *moved_out = 0;
    std::lock_guard<std::mutex> g(d->mu);
    Index* hd = d->head;
    std::lock_guard<std::mutex> gh(hd->mu);
    if (hd->last_stream) CK(cudaStreamSynchronize(hd->last_stream));
    Segment& hs = hd->seg;
    const int64_t n = do_move ? hs.live : 0;
    if (d->stail) {
        // sharded tail: the rows are gathered once on the head's device; every shard copies them over (peer copies)
        // and applies the same step to its replica of the buffer and to the lists it owns
        if (n > 0) {
            DevBuf mx, ml;
            std::vector<int64_t> mlab;
            TRY(gather_head_rows(hd, n, mx, ml, mlab, hd->stream));
            TRY(pyrope_internal_sharded_absorb(d->stail, n, mx.as<float>(), ml.as<int64_t>(), hd->device, mlab.data(),
                                               tail_rows_out));
        }
    } else {
        Index* tl = d->tail;
        std::lock_guard<std::mutex> gt(tl->mu);
        if (tl->last_stream) CK(cudaStreamSynchronize(tl->last_stream));
        if (n > 0) {
            DevBuf mx, ml;
            std::vector<int64_t> mlab;
            TRY(gather_head_rows(hd, n, mx, ml, mlab, tl->stream));
            TRY(tail_absorb(tl, n, mx.as<float>(), ml.as<int64_t>(), mlab.data(), tail_rows_out));
        }
    }
    if (n > 0) {
        // 3. _head.Delete(id) per row (:147): tombstones, slots stay (BruteForceVectorIndex.cs:231-254)
        CK(cudaMemsetAsync(hs.dead.p, 1, (size_t)hs.nslots, hd->stream));
        std::fill(hs.dead_h.begin(), hs.dead_h.end(), (uint8_t)1);
        hs.ndead = hs.nslots;
        hs.live = 0;
        hs.tc_dirty = true;
        CK(cudaStreamSynchronize(hd->stream));
        if (moved_out) *moved_out = n;
    }
    // 4. _head.Build() is a no-op for FLAT; _tail.Build() (:151-152)
    if (!do_build) return PYROPE_OK;
    if (d->stail) return extend ? pyrope_sharded_extend(d->stail) : pyrope_sharded_build(d->stail);
    Index* tl = d->tail;
    std::lock_guard<std::mutex> gt(tl->mu);
    Staged S(*tl);
    TRY(extend ? extend_prepare(*tl, S) : build_prepare(*tl, S));
    install(tl, S);
    return PYROPE_OK;
}
}  // namespace

extern "C" {

// ---- internal (not in the public header): the compaction's per-tail step for csrc/sharded.cu, run on each shard's
// thread.  _reserve makes room for n more buffer rows before any shard writes; _absorb is tail_absorb above.
int pyrope_internal_tail_reserve(pyrope_index* tl, int64_t n) {
    if (!tl || n < 0) return fail(PYROPE_ERR_INVALID_ARG, "bad argument");
    std::lock_guard<std::mutex> g(tl->mu);
    TRY(tl->seg.reserve(tl->seg.nslots + n, tl->stream, false));
    CK(cudaStreamSynchronize(tl->stream));
    return PYROPE_OK;
}

int pyrope_internal_tail_absorb(pyrope_index* tl, int64_t n, const float* dX, const int64_t* dL, const int64_t* labels_host,
                                int64_t* tail_rows_out) {
    if (!tl || n < 0 || (n > 0 && (!dX || !dL || !labels_host))) return fail(PYROPE_ERR_INVALID_ARG, "bad argument");
    std::lock_guard<std::mutex> g(tl->mu);
    if (tl->last_stream) CK(cudaStreamSynchronize(tl->last_stream));
    if (n == 0) return PYROPE_OK;
    return tail_absorb(tl, n, dX, dL, labels_host, tail_rows_out);
}

int pyrope_delta_compact(pyrope_delta* d, int64_t* moved_out, int64_t* tail_rows_out) {
    return delta_compact_impl(d, moved_out, tail_rows_out, true, true);
}
int pyrope_delta_move(pyrope_delta* d, int64_t* moved_out, int64_t* tail_rows_out) {
    return delta_compact_impl(d, moved_out, tail_rows_out, true, false);
}
int pyrope_delta_build_tail(pyrope_delta* d) { return delta_compact_impl(d, nullptr, nullptr, false, true); }
int pyrope_delta_extend_tail(pyrope_delta* d) { return delta_compact_impl(d, nullptr, nullptr, false, true, true); }

int pyrope_delta_stats(pyrope_delta* d, int64_t* count_out) {
    if (!d || !count_out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    // DeltaVectorIndex.cs:232-236: plain sum of both sides (duplicates counted twice, as in the reference)
    Index* hd = d->head;
    if (d->stail) {
        int64_t t = 0;
        TRY(pyrope_sharded_stats(d->stail, &t));
        *count_out = hd->seg.live + t;
        return PYROPE_OK;
    }
    Index* tl = d->tail;
    *count_out = hd->seg.live + tl->seg.live + (tl->built ? tl->lists.total - tl->lists.ndead : 0);
    return PYROPE_OK;
}

int pyrope_delta_snapshot(pyrope_delta* d, const char* path) {
    if (!d) return fail(PYROPE_ERR_INVALID_ARG, "delta handle is null");
    if (!path || !*path) return fail(PYROPE_ERR_INVALID_ARG, "Path cannot be empty.");
    const std::string base(path);
    TRY(pyrope_index_snapshot(d->head, (base + ".head").c_str()));
    if (d->stail) TRY(pyrope_sharded_snapshot(d->stail, (base + ".tail").c_str()));
    else TRY(pyrope_index_snapshot(d->tail, (base + ".tail").c_str()));
    const std::string tmp = base + ".tmp";
    FILE* f = fopen(tmp.c_str(), "wb");
    if (!f) return fail(PYROPE_ERR_INVALID_ARG, "cannot open %s for writing", tmp.c_str());
    const char* manifest = "{\"Type\": \"Delta\", \"Head\": \".head\", \"Tail\": \".tail\"}";  // DeltaVectorIndex.cs:183
    const bool ok = fwrite(manifest, 1, strlen(manifest), f) == strlen(manifest);
    if (fclose(f) != 0 || !ok) { remove(tmp.c_str()); return fail(PYROPE_ERR_INVALID_ARG, "short write to %s", tmp.c_str()); }
    if (rename(tmp.c_str(), base.c_str()) != 0) { remove(tmp.c_str()); return fail(PYROPE_ERR_INVALID_ARG, "cannot move %s into place", tmp.c_str()); }
    return PYROPE_OK;
}

int pyrope_delta_load(pyrope_delta* d, const char* path) {
    if (!d) return fail(PYROPE_ERR_INVALID_ARG, "delta handle is null");
    if (!path || !*path) return fail(PYROPE_ERR_INVALID_ARG, "Path cannot be empty.");
    const std::string base(path);
    // DeltaVectorIndex.cs:200-216: each side is loaded only if its file exists
    for (int side = 0; side < 2; ++side) {
        const std::string p = base + (side == 0 ? ".head" : ".tail");
        FILE* f = fopen(p.c_str(), "rb");
        if (!f) continue;
        fclose(f);
        if (side == 1 && d->stail) TRY(pyrope_sharded_load(d->stail, p.c_str()));
        else TRY(pyrope_index_load(side == 0 ? d->head : d->tail, p.c_str()));
    }
    return PYROPE_OK;
}

// ---- building blocks (host pointers) -------------------------------------------------------------
int pyrope_coarse_assign(int metric, int dim, int64_t n, const float* X, int n_centroids, const float* centroids,
                         int32_t* assign_out) {
    if (!X || !centroids || !assign_out || dim <= 0 || n < 0 || n_centroids <= 0)
        return fail(PYROPE_ERR_INVALID_ARG, "bad arguments");
    TRY(ensure_init());
    if (n == 0) return PYROPE_OK;
    DevBuf dx, dc, dn, da;
    cudaStream_t st = nullptr;
    TRY(dx.ensure(sizeof(float) * (size_t)n * dim, 0, st, true));
    TRY(dc.ensure(sizeof(float) * (size_t)n_centroids * dim, 0, st, true));
    TRY(dn.ensure(sizeof(float) * (size_t)n_centroids, 0, st, true));
    TRY(da.ensure(sizeof(int32_t) * (size_t)n, 0, st, true));
    CK(cudaMemcpy(dx.p, X, sizeof(float) * (size_t)n * dim, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dc.p, centroids, sizeof(float) * (size_t)n_centroids * dim, cudaMemcpyHostToDevice));
    if (metric == kCosine) CK(launch_row_norms_exact(dc.as<float>(), n_centroids, dim, dim, dn.as<float>(), st));
    AssignScratch as;
    TRY(assign_rows(metric, dim, n, dx.as<float>(), dim, n_centroids, dc.as<float>(), dn.as<float>(), da.as<int32_t>(), as, true, st));
    CK(cudaMemcpy(assign_out, da.p, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost));
    return PYROPE_OK;
}

int pyrope_kmeans_train(int metric, int dim, int64_t n, int64_t ld, const float* data, int k, int max_iter, int32_t seed,
                        float* centroids_out, int* k_out, int* iters_out) {
    if (!data || !centroids_out || !k_out || dim <= 0 || n < 0 || ld < dim) return fail(PYROPE_ERR_INVALID_ARG, "bad arguments");
    TRY(ensure_init());
    *k_out = 0;
    if (n == 0) return PYROPE_OK;
    int kk = k <= 0 ? 1 : (int)std::min<int64_t>(k, n);
    DevBuf dx, dc;
    cudaStream_t st = nullptr;
    TRY(dx.ensure(sizeof(float) * (size_t)n * ld, 0, st, true));
    TRY(dc.ensure(sizeof(float) * (size_t)kk * dim, 0, st, true));
    CK(cudaMemcpy(dx.p, data, sizeof(float) * (size_t)n * ld, cudaMemcpyHostToDevice));
    TRY(kmeans_train_device(metric, dim, n, ld, dx.as<float>(), k, max_iter, seed, dc.as<float>(), k_out, iters_out, st));
    CK(cudaMemcpy(centroids_out, dc.p, sizeof(float) * (size_t)(*k_out) * dim, cudaMemcpyDeviceToHost));
    return PYROPE_OK;
}

int pyrope_pq_encode(int dim, int m, int k, const float* codebooks, const int32_t* ksub, int64_t n, const float* X,
                     uint8_t* codes_out) {
    if (!codebooks || !X || !codes_out || dim <= 0 || m <= 0 || dim % m || k <= 0 || k > 256 || n < 0)
        return fail(PYROPE_ERR_INVALID_ARG, "bad arguments");
    TRY(ensure_init());
    if (n == 0) return PYROPE_OK;
    DevBuf dx, dc, dk, dcode;
    cudaStream_t st = nullptr;
    const int sub = dim / m;
    TRY(dx.ensure(sizeof(float) * (size_t)n * dim, 0, st, true));
    TRY(dc.ensure(sizeof(float) * (size_t)m * k * sub, 0, st, true));
    TRY(dk.ensure(sizeof(int32_t) * (size_t)m, 0, st, true));
    TRY(dcode.ensure((size_t)n * m, 0, st, true));
    std::vector<int32_t> ks((size_t)m, k);
    if (ksub) memcpy(ks.data(), ksub, sizeof(int32_t) * (size_t)m);
    CK(cudaMemcpy(dx.p, X, sizeof(float) * (size_t)n * dim, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dc.p, codebooks, sizeof(float) * (size_t)m * k * sub, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dk.p, ks.data(), sizeof(int32_t) * (size_t)m, cudaMemcpyHostToDevice));
    CK(launch_pq_encode_exact(dx.as<float>(), n, dim, m, k, dc.as<float>(), dk.as<int32_t>(), dcode.as<uint8_t>(), st));
    CK(cudaMemcpy(codes_out, dcode.p, (size_t)n * m, cudaMemcpyDeviceToHost));
    return PYROPE_OK;
}

int pyrope_pq_distance_table(int dim, int m, int k, const float* codebooks, int64_t nq, const float* Q, float* table_out) {
    if (!codebooks || !Q || !table_out || dim <= 0 || m <= 0 || dim % m || k <= 0 || nq < 0)
        return fail(PYROPE_ERR_INVALID_ARG, "bad arguments");
    TRY(ensure_init());
    if (nq == 0) return PYROPE_OK;
    DevBuf dq, dc, dt;
    cudaStream_t st = nullptr;
    TRY(dq.ensure(sizeof(float) * (size_t)nq * dim, 0, st, true));
    TRY(dc.ensure(sizeof(float) * (size_t)k * dim, 0, st, true));
    TRY(dt.ensure(sizeof(float) * (size_t)nq * m * k, 0, st, true));
    CK(cudaMemcpy(dq.p, Q, sizeof(float) * (size_t)nq * dim, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dc.p, codebooks, sizeof(float) * (size_t)k * dim, cudaMemcpyHostToDevice));
    CK(launch_pq_distance_table(dq.as<float>(), nq, dim, dc.as<float>(), m, k, dt.as<float>(), st));
    CK(cudaMemcpy(table_out, dt.p, sizeof(float) * (size_t)nq * m * k, cudaMemcpyDeviceToHost));
    return PYROPE_OK;
}

int pyrope_fill_uniform_device(float* d_out, int64_t n, uint64_t seed, uint64_t offset, void* stream) {
    if (!d_out || n < 0) return fail(PYROPE_ERR_INVALID_ARG, "bad arguments");
    CK(launch_fill_uniform(d_out, n, seed, offset, (cudaStream_t)stream));
    return PYROPE_OK;
}

}  // extern "C"
