// peer.cu — the exchange step of the sharded search (SURVEY §8e: every GPU emits per-query data, every GPU needs all
// of it) written directly over NVLink peer memory instead of through a collective library.
//
// A pyrope_peer_group is one rank's end of an N-way all-gather: a device buffer the PEERS write into (mapped into their
// address spaces through CUDA IPC when every rank is its own process, or handed over as plain device pointers when one
// process drives all GPUs) plus a few flag words.  pyrope_peer_allgather_device() runs entirely on the caller's stream:
//   1. peer_scatter_kernel   copies this rank's contribution into slot [rank] of EVERY rank's buffer (16-byte peer
//                            stores, one block column per destination so all NVLink ports are busy at once);
//   2. peer_signal_wait_kernel  writes this call's epoch into every peer's flag word for this rank (after a
//                            system-scope fence) and then polls its own flag words until every peer's epoch arrived.
// No host round trip, no second stream, no library: two small launches (~10 us) where an NCCL all-gather of the same
// few megabytes costs ~45 us per call in this pipeline (bench.py, step_phases_ms).
//
// Reuse: the data area of a slot is double-buffered by epoch parity.  A rank can start call n+1 as soon as its own call
// n returned, i.e. as soon as every peer SIGNALLED call n — the peer may still be reading call n's data, which lives in
// the other half.  It cannot start call n+2 before every peer signalled n+1, and a peer signals n+1 in stream order
// after everything it launched between its calls n and n+1 — so the consumers of call n's data must be launched on the
// same stream, before the next call, which is how a search step uses it.
// Every rank must issue the same sequence of calls (slot, size): the epoch is a per-slot call counter.
#include <algorithm>
#include <cstring>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/pyrope_gpu.h"
#include "internal.h"

namespace {

constexpr int kMaxWorld = 8;
constexpr int kMaxSlots = 8;
constexpr size_t kFlagBytes = 4096;  // [kMaxSlots][kMaxWorld] 64-bit epoch words at the head of the allocation

struct PeerPtrs {
    unsigned char* base[kMaxWorld];
};

// grid (chunks, world): block column r copies src into rank r's buffer at dst_off
__global__ void __launch_bounds__(256) peer_scatter_kernel(PeerPtrs pp, size_t dst_off, const uint4* __restrict__ src, size_t n16) {
    uint4* dst = reinterpret_cast<uint4*>(pp.base[blockIdx.y] + dst_off);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) dst[i] = __ldg(src + i);
}

// one block, one thread per rank: publish my epoch at rank r, then wait for rank r's epoch here
__global__ void peer_signal_wait_kernel(PeerPtrs pp, int world, int rank, int slot, unsigned long long epoch) {
    const int r = threadIdx.x;
    if (r < world && r != rank) {
        __threadfence_system();  // the scatter kernel's stores (already complete: stream order) and anything else before the flag
        volatile unsigned long long* theirs =
            reinterpret_cast<volatile unsigned long long*>(pp.base[r]) + (size_t)slot * kMaxWorld + rank;
        *theirs = epoch;
        volatile unsigned long long* mine =
            reinterpret_cast<volatile unsigned long long*>(pp.base[rank]) + (size_t)slot * kMaxWorld + r;
        unsigned long long spins = 0;
        while (*mine < epoch) {
            __nanosleep(200);
            if (++spins > (1ull << 26)) __trap();  // ~20 s: a peer that never arrives must fault, not hang the GPU
        }
        __threadfence_system();
    }
}

}  // namespace

struct pyrope_peer_group {
    int world = 0, rank = 0, device = 0;
    size_t slot_bytes = 0;  // per rank, per slot, per parity half
    int n_slots = 0;
    size_t total = 0;
    unsigned char* local = nullptr;
    unsigned char* peers[kMaxWorld] = {nullptr};
    bool attached = false, ipc = false;
    unsigned long long epoch[kMaxSlots] = {0};
};

extern "C" {

int pyrope_peer_group_create(int world, int rank, size_t slot_bytes, int n_slots, pyrope_peer_group** out) {
    if (!out) return fail(PYROPE_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    if (world < 2 || world > kMaxWorld || rank < 0 || rank >= world) return fail(PYROPE_ERR_INVALID_ARG, "world must be 2..8, rank below it");
    if (n_slots < 1 || n_slots > kMaxSlots || slot_bytes == 0) return fail(PYROPE_ERR_INVALID_ARG, "1..8 slots of at least one byte");
    pyrope_peer_group* g = new (std::nothrow) pyrope_peer_group();
    if (!g) return fail(PYROPE_ERR_OOM, "out of host memory");
    g->world = world; g->rank = rank; g->n_slots = n_slots;
    g->slot_bytes = (slot_bytes + 255) & ~(size_t)255;
    g->total = kFlagBytes + (size_t)n_slots * 2 * world * g->slot_bytes;
    cudaError_t e = cudaGetDevice(&g->device);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&g->local), g->total);
    if (e == cudaSuccess) e = cudaMemset(g->local, 0, kFlagBytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        const size_t want = g->total;
        if (g->local) cudaFree(g->local);
        delete g;
        return fail(e == cudaErrorMemoryAllocation ? PYROPE_ERR_OOM : PYROPE_ERR_CUDA, "peer group buffer (%zu bytes): %s", want,
                    cudaGetErrorString(e));
    }
    g->peers[rank] = g->local;
    *out = g;
    return PYROPE_OK;
}

int pyrope_peer_group_destroy(pyrope_peer_group* g) {
    if (!g) return PYROPE_OK;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(g->device);
    cudaDeviceSynchronize();
    if (g->ipc)
        for (int r = 0; r < g->world; ++r)
            if (r != g->rank && g->peers[r]) cudaIpcCloseMemHandle(g->peers[r]);
    if (g->local) cudaFree(g->local);
    if (prev >= 0) cudaSetDevice(prev);  // the caller's current device is not ours to change
    delete g;
    return PYROPE_OK;
}

int pyrope_peer_group_handle(pyrope_peer_group* g, void* handle_out) {
    if (!g || !handle_out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    cudaIpcMemHandle_t hd;
    CK(cudaIpcGetMemHandle(&hd, g->local));
    memcpy(handle_out, &hd, sizeof hd);
    return PYROPE_OK;
}

int pyrope_peer_group_buffer(pyrope_peer_group* g, void** d_buffer_out) {
    if (!g || !d_buffer_out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    *d_buffer_out = g->local;
    return PYROPE_OK;
}

int pyrope_peer_group_open(pyrope_peer_group* g, const void* handles) {
    if (!g || !handles) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    if (g->attached) return fail(PYROPE_ERR_INVALID_STATE, "peers are already attached");
    for (int r = 0; r < g->world; ++r) {
        if (r == g->rank) continue;
        cudaIpcMemHandle_t hd;
        memcpy(&hd, static_cast<const unsigned char*>(handles) + (size_t)r * sizeof hd, sizeof hd);
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            for (int rr = 0; rr < r; ++rr)
                if (rr != g->rank && g->peers[rr]) { cudaIpcCloseMemHandle(g->peers[rr]); g->peers[rr] = nullptr; }
            return fail(PYROPE_ERR_UNSUPPORTED, "cannot map the buffer of rank %d: %s", r, cudaGetErrorString(e));
        }
        g->peers[r] = static_cast<unsigned char*>(p);
    }
    g->attached = true;
    g->ipc = true;
    return PYROPE_OK;
}

int pyrope_peer_group_attach(pyrope_peer_group* g, void* const* buffers) {
    if (!g || !buffers) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    if (g->attached) return fail(PYROPE_ERR_INVALID_STATE, "peers are already attached");
    for (int r = 0; r < g->world; ++r) {
        if (r == g->rank) continue;
        if (!buffers[r]) return fail(PYROPE_ERR_INVALID_ARG, "buffer of rank %d is null", r);
        g->peers[r] = static_cast<unsigned char*>(buffers[r]);
    }
    g->attached = true;
    g->ipc = false;
    return PYROPE_OK;
}

int pyrope_peer_allgather_device(pyrope_peer_group* g, int slot, const void* d_src, size_t bytes_per_rank, const void** d_gathered_out,
                                 void* stream) {
    if (!g || !d_src || !d_gathered_out) return fail(PYROPE_ERR_INVALID_ARG, "null argument");
    if (!g->attached) return fail(PYROPE_ERR_INVALID_STATE, "attach or open the peers first");
    if (slot < 0 || slot >= g->n_slots) return fail(PYROPE_ERR_INVALID_ARG, "slot %d of %d", slot, g->n_slots);
    if (bytes_per_rank == 0 || bytes_per_rank > g->slot_bytes || (bytes_per_rank & 15) || (reinterpret_cast<uintptr_t>(d_src) & 15))
        return fail(PYROPE_ERR_INVALID_ARG, "contribution must be 16-byte aligned, a multiple of 16 bytes and at most %zu bytes", g->slot_bytes);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned long long epoch = g->epoch[slot] + 1;  // committed below, once both kernels are enqueued
    // [slot][parity][rank][bytes_per_rank]: the ranks' contributions are contiguous, like an all-gather's output
    const size_t half = kFlagBytes + ((size_t)slot * 2 + (epoch & 1)) * g->world * g->slot_bytes;
    PeerPtrs pp{};
    for (int r = 0; r < g->world; ++r) pp.base[r] = g->peers[r];
    const size_t n16 = bytes_per_rank / 16;
    const unsigned chunks = (unsigned)std::min<size_t>(32, (n16 + 255) / 256);
    peer_scatter_kernel<<<dim3(chunks, (unsigned)g->world), 256, 0, st>>>(pp, half + (size_t)g->rank * bytes_per_rank,
                                                                        static_cast<const uint4*>(d_src), n16);
    peer_signal_wait_kernel<<<1, 32, 0, st>>>(pp, g->world, g->rank, slot, epoch);
    CK(cudaGetLastError());
    g->epoch[slot] = epoch;
    *d_gathered_out = g->local + half;
    return PYROPE_OK;
}

}  // extern "C"
